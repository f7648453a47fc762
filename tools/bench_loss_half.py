#!/usr/bin/env python
"""K4 on fp16 / bf16 logits against the fp32 routes a mixed-precision training step can take, at B = 64, K = 5, 256 x 480,
with uint8 and with int64 targets.  One JSON line per variant:

  a      fp32 K4, forward+backward in one launch (today's fp32 training step)
  b      the AMP workaround: cast the half logits up, fp32 K4, scale the gradients by 2^16 as a GradScaler's backward does
         (mspl_scale_inplace), cast them back down
  c      fp16 / bf16 K4, forward+backward in one launch (ops.uw_ce_fwd_bwd)
  c_fwd  fp16 / bf16 K4, forward only (the first half of d)
  d      fp16 / bf16 through autograd (ops.uw_ce_loss): forward-only launch, then backward with the upstream scale 1 or 2^16

All variants are timed alternately in one process, with the L2 flushed (a 256 MiB write) before every timed step; ms is the
median of --steps steps after --warmup.  bytes_per_px is what the algorithm has to move per pixel, computed from the shapes;
frac_of_copy_peak divides the achieved rate by a device-to-device copy measured in the same run.  Card name and power limit
are read in the same run.

  python tools/bench_loss_half.py [--steps 50] [--warmup 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mspl_b200 import _lib, ops  # noqa: E402


def power_limit_w(index):
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(index)],
                                      text=True, timeout=30)
        return float(out.strip().splitlines()[0])
    except (OSError, subprocess.SubprocessError, ValueError, IndexError):
        return None


def copy_peak_gbs(dev, steps=20):
    """Device-to-device copy of 2 GiB (read + write counted), median over `steps`."""
    src = torch.empty(2 ** 31, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    ms = []
    for i in range(steps + 3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(src)
        e1.record()
        torch.cuda.synchronize()
        if i >= 3:
            ms.append(e0.elapsed_time(e1))
    ms.sort()
    del src, dst
    return 2 * 2 ** 31 / 1e9 / (ms[len(ms) // 2] / 1e3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    card = torch.cuda.get_device_name(dev)
    power = power_limit_w(dev.index)
    b, k, h, w = 64, 5, 256, 480
    pix = b * h * w
    peak = copy_peak_gbs(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    cw = torch.tensor([1.0, 1.0, 1.0, 1.0, 0.0], device=dev)
    g = torch.Generator(device=dev).manual_seed(11)
    main32 = 3 * torch.randn((b, k, h, w), device=dev, generator=g)
    aux32 = main32 + 1.5 * torch.randn((b, k, h, w), device=dev, generator=g)
    tgt64 = torch.randint(1, 5, (b, h, w), device=dev, generator=g)
    halves = {dt: (main32.to(dt), aux32.to(dt)) for dt in (torch.bfloat16, torch.float16)}
    scale_dev = torch.tensor([2.0 ** 16], device=dev)
    lib = _lib.load()

    def scale_inplace(x):
        _lib.check(lib.mspl_scale_inplace(ops._ptr(x), x.numel(), ops._ptr(scale_dev), ops._stream(dev)), "mspl_scale_inplace")

    variants = []            # (name, dtype name, target name, bytes per pixel, fn)
    for tname, tgt in (("u8", tgt64.to(torch.uint8)), ("int64", tgt64)):
        tb = tgt.element_size()
        variants.append(("a_fp32_one_launch", "fp32", tname, 2 * 4 * k * 2 + tb,
                         lambda t=tgt: ops.uw_ce_fwd_bwd(main32, aux32, t, cw)))
        for dt, (mh, ah) in halves.items():
            dn = str(dt).replace("torch.", "")

            def amp_workaround(mh=mh, ah=ah, t=tgt, dt=dt):
                out3, dm, da = ops.uw_ce_fwd_bwd(mh.float(), ah.float(), t, cw)
                scale_inplace(dm)
                scale_inplace(da)
                return out3, dm.to(dt), da.to(dt)
            # casts up (2 B read, 4 B written per logit), fp32 K4, two scale passes (4 B read + 4 B written), casts down (4 + 2)
            variants.append(("b_amp_workaround_scale65536", dn, tname, 2 * k * 6 + (2 * 4 * k * 2 + tb) + 2 * k * 8 + 2 * k * 6,
                             amp_workaround))
            variants.append(("c_half_one_launch", dn, tname, 2 * 2 * k * 2 + tb, lambda mh=mh, ah=ah, t=tgt: ops.uw_ce_fwd_bwd(mh, ah, t, cw)))
            variants.append(("c_fwd_half_forward_only", dn, tname, 2 * 2 * k + tb,
                             lambda mh=mh, ah=ah, t=tgt: ops.uw_ce_fwd_bwd(mh, ah, t, cw, backward=False)))
            for s in (1.0, 2.0 ** 16):
                leaves = (mh.clone().requires_grad_(True), ah.clone().requires_grad_(True))

                def autograd_step(leaves=leaves, t=tgt, s=s):
                    m, a = leaves
                    m.grad = a.grad = None
                    loss = ops.uw_ce_loss(m, a, t, cw)
                    (loss if s == 1.0 else loss * s).backward()
                    return loss
                variants.append(("d_half_autograd_scale%d" % s, dn, tname, (2 * 2 * k + tb) + (2 * 2 * k * 2 + tb), autograd_step))

    for _ in range(args.warmup):
        for v in variants:
            v[4]()
    torch.cuda.synchronize()
    times = [[] for _ in variants]
    for _ in range(args.steps):
        for i, v in enumerate(variants):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            v[4]()
            e1.record()
            torch.cuda.synchronize()
            times[i].append(e0.elapsed_time(e1))
    lines = []
    for (name, dn, tname, bpp, _), ms in zip(variants, times):
        ms.sort()
        med = ms[len(ms) // 2]
        gbs = pix * bpp / 1e9 / (med / 1e3)
        lines.append(json.dumps({"name": name, "logits": dn, "target": tname, "B": b, "K": k, "H": h, "W": w,
                                 "ms_median": round(med, 4), "ms_min": round(ms[0], 4), "steps": args.steps,
                                 "bytes_per_px": bpp, "GB/s": round(gbs, 1), "frac_of_copy_peak": round(gbs / peak, 3),
                                 "copy_peak_GB/s": round(peak, 1), "card": card, "power_limit_W": power,
                                 "lib": os.path.relpath(_lib.LIB_PATH, ROOT),
                                 "note": "L2 flushed before every timed step; variants alternated"}))
    for line in lines:
        print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
