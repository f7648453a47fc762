#!/usr/bin/env python
"""Benchmark of the hot path: 3-source pseudo-label generation (Cityscapes/CamVid/Forest logits -> greenhouse classes)
with class-balanced thresholds.

  python bench.py --gpus N --steps K --warmup W              (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W    (CPU reference arm, rank 0 only)
  python bench.py ... --dump-outputs DIR                      (also write the last timed step's outputs as DIR/*.npy)

Workload (BASELINE.json configs): N = 1 runs configs[1], 2,000 synthetic 480x256 images resident in HBM; N > 1 runs configs[2],
a 20,000-image target set sharded by contiguous image range over the ranks (strong scaling: 10,000 / 5,000 / 2,500 images per
GPU).  A shard larger than HBM holds as logits is labelled by cycling a resident 2,500-image pool (image i of the set = pool
image i mod 2,500, the same pool on every rank, so the set -- and the digest of its thresholds and histograms -- does not
depend on the rank count); label / confidence / uncertainty maps and all statistics are those of the full shard.
A "step" is one whole pass of the path over this rank's shard: K1 fuse_sources per pool cycle (+ linear confidence histogram)
-> [one all-reduce of the packed statistics] -> bracket select -> one classify pass -> candidate radix select (one launch on
a single rank; three histogram all-reduces under N ranks).  `value` = pixels labelled by all ranks / max-over-ranks device time.
`e2e` = the same metric through the public host-buffer API (LabelGenerator.run_from_host): pinned host logits -> H2D ->
kernels -> D2H of the uint8 label maps, all inside the timed region, next to the bare host-to-device copy ceiling measured
concurrently on all ranks.  `roofline` is the fused kernel K1 alone (CUDA events around each launch, live) against the
measured HBM peak in MEASURED_PEAKS.json.  `cpu_baseline` / `--impl reference` time the reference's OWN functions (staged by
oracle/build_ref.py under oracle/_ref; the oracle port if absent) on a bounded sample.  `secondary` carries the other
configurations north_star names, each with its own roofline and checks: the per-class K1 policies, the 20,000-image set on one
GPU, the uncertainty-weighted loss (configs[3]), the 1024x512 stress case (configs[4]) and the fused-upsample kernel.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SOURCES = (("camvid", 13), ("cityscapes", 20), ("forest", 5))
SIGMA = 3.0
FALLBACK_HBM_GBS = 6650.0     # /opt/skills/guides/B200_PROFILING.md fallback, used only if MEASURED_PEAKS.json is absent
POOL_IMAGES = 2500            # resident logits per rank: 93.4 GB at 480x256 (configs[2] at 8 GPUs is exactly one pool)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=("native", "reference"), default="native")
    ap.add_argument("--images-total", type=int, default=0,
                    help="target images over all ranks; 0 = configs[1] (2,000) on one GPU, configs[2] (20,000) on several")
    ap.add_argument("--height", type=int, default=256)
    ap.add_argument("--width", type=int, default=480)
    ap.add_argument("--policy", default="all", help="espdnet_greenhouse_uest_multi_os.sh: --merge-label-policy all")
    ap.add_argument("--portion", type=float, default=0.2, help="INIT_TGT_PORT (uest_seg_multi_os.py:90)")
    ap.add_argument("--e2e-images", type=int, default=128, help="images per end-to-end step (host buffers)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU baseline budget (bounded sample)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--ref-images", type=int, default=32, help="--impl reference: images per step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy: rank 0 writes the global statistics "
                         "and a seeded sample of its own shard's maps (see dump_outputs); --impl reference writes the "
                         "class weights")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def images_total(args, world):
    return args.images_total if args.images_total > 0 else (2000 if world == 1 else 20000)


# ---- synthetic inputs (SURVEY.md 8d): main = sigma*randn + per-image class bias; aux = main + 0.5*sigma*randn ----------
def make_logits_device(torch, n, h, w, device, seed, sources=SOURCES, chunk=50, lowres=False):
    gen = torch.Generator(device=device).manual_seed(seed)
    mains, auxs = [], []
    for _, c in sources:
        ms = (n, c, h // 2, w // 2) if lowres else (n, c, h, w)
        as_ = (n, c, h // 4, w // 4) if lowres else (n, c, h, w)
        m = torch.empty(ms, dtype=torch.float32, device=device)
        a = torch.empty(as_, dtype=torch.float32, device=device)
        for lo in range(0, n, chunk):
            hi = min(n, lo + chunk)
            m[lo:hi].normal_(0.0, SIGMA, generator=gen)
            m[lo:hi] += SIGMA * torch.randn((hi - lo, c, 1, 1), device=device, generator=gen)
            a[lo:hi].normal_(0.0, 0.5 * SIGMA, generator=gen)
            if lowres:
                a[lo:hi] += torch.nn.functional.avg_pool2d(m[lo:hi], 2)
            else:
                a[lo:hi] += m[lo:hi]
        mains.append(m), auxs.append(a)
    return mains, auxs


def make_logits_host(torch, n, h, w, seed, pin, lowres=False):
    gen = torch.Generator().manual_seed(seed)
    mains, auxs = [], []
    for _, c in SOURCES:
        if lowres:
            m = SIGMA * torch.randn((n, c, h // 2, w // 2), generator=gen) + SIGMA * torch.randn((n, c, 1, 1), generator=gen)
            a = torch.nn.functional.avg_pool2d(m, 2) + 0.5 * SIGMA * torch.randn((n, c, h // 4, w // 4), generator=gen)
        else:
            m = SIGMA * torch.randn((n, c, h, w), generator=gen) + SIGMA * torch.randn((n, c, 1, 1), generator=gen)
            a = m + 0.5 * SIGMA * torch.randn((n, c, h, w), generator=gen)
        mains.append(m.pin_memory() if pin else m), auxs.append(a.pin_memory() if pin else a)
    return mains, auxs


# ---- clocks during the timed region (B200_PROFILING.md) ---------------------------------------------------------------
class ClockSampler:
    """nvidia-smi polled every 20 ms from process start; stop(t0, t1) keeps the samples taken inside the timed region."""
    QUERY = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_ms=20):
        self.index, self.proc, self.lines, self.period_ms = index, None, [], int(period_ms)

    def start(self):
        if self.period_ms <= 0:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self, t0, t1):
        import datetime
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        rows = []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), float(f[2]), float(f[3]), [nm for nm, v in zip(names, f[5:9]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        inside = [r for r in rows if t0 <= r[0] <= t1]
        window = "timed region"
        if len(inside) < 3:      # very short timed region: widen to the neighbouring samples and say so
            inside = [r for r in rows if t0 - 0.25 <= r[0] <= t1 + 0.1]
            window = "timed region +-0.25 s (region shorter than 3 samples)"
        sm = sorted(r[1] for r in inside)
        reasons = sorted({nm for r in inside for nm in r[4]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max((r[2] for r in inside), default=None),
                "power_w_max": max((r[3] for r in inside), default=None), "samples": len(inside), "window": window,
                "reasons": reasons}


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one K1 launch from the committed ncu capture, if any."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "k1_traffic.json")))
    except Exception:
        return None


# ---- CPU arm: the reference's own functions (oracle/_ref or /root/reference), else the oracle port ----------------------
class CpuPath:
    """One image after the other through get_output -> argmax -> id_*_to_greenhouse -> merge_outputs -> class_array, composed
    exactly as the reference's loop does (uest_seg_multi_os.py:888-950)."""

    def __init__(self):
        from oracle import ref_import
        self.ref = None
        try:
            self.ref = ref_import.load_reference(allow_staged=True)
        except Exception as exc:          # a broken staging must not take the bench down: fall back to the port and say so
            self.error = "%s: %s" % (type(exc).__name__, exc)
        from oracle import mspl_oracle as O
        self.O = O
        self.FixedLogitsModel = ref_import.FixedLogitsModel
        self.kind = "reference" if self.ref is not None else "port"
        if self.ref is not None:
            g = self.ref.greenhouse
            self.tables = {"camvid": g.id_camvid_to_greenhouse, "cityscapes": g.id_cityscapes_to_greenhouse,
                           "forest": g.id_forest_to_greenhouse}
        self.luts = [O.LUTS[s] for s, _ in SOURCES]

    def describe(self):
        if self.kind == "reference":
            return ("the reference's own get_output / merge_outputs / id_*_to_greenhouse (uest_seg_multi_os.py:669-718, 897-921; "
                    "files staged by oracle/build_ref.py, origin=%s)" % self.ref.origin)
        return "oracle port of get_output->argmax->LUT->merge_outputs->class_array (uest_seg_multi_os.py:897-921); oracle/_ref not staged"

    def images(self, torch, np, mains, auxs, policy, lo, hi):
        """Label images [lo, hi): returns class_array (K,) float64."""
        if self.kind == "port":
            _, class_array = self.O.multi_source_labels([m[lo:hi] for m in mains], [a[lo:hi] for a in auxs], self.luts, policy)
            return class_array
        U = self.ref.uest
        class_array = np.zeros(5)
        dummy = torch.zeros(1, 3, 1, 1)
        with torch.no_grad():
            for i in range(lo, hi):
                output_list = []
                for s, (name, _) in enumerate(SOURCES):
                    output, _ = U.get_output(self.FixedLogitsModel(mains[s][i:i + 1], auxs[s][i:i + 1]), dummy, device='cpu')
                    output = output.transpose(1, 2, 0)
                    amax_output = np.asarray(np.argmax(output, axis=2), dtype=np.uint8)
                    output_list.append(self.tables[name][amax_output])
                amax_output = U.merge_outputs(np.array(output_list), seg_classes=5, thresh=policy)
                for k in range(5):
                    class_array[k] += (amax_output == k).sum()
        return class_array

    def step(self, torch, np, mains, auxs, policy, pool=None, workers=1):
        """All images of the batch; with a pool the images are dealt to `workers` host threads (torch's CPU ops release the
        GIL) -- the reference's loop is sequential and only gets torch's intra-op threads, which the small per-image tensors
        do not fill, so this is the arrangement that uses every host core."""
        n = mains[0].shape[0]
        if pool is None:
            class_array = self.images(torch, np, mains, auxs, policy, 0, n)
        else:
            class_array = sum(pool.map(lambda i: self.images(torch, np, mains, auxs, policy, i, i + 1), range(n)))
        return self.O.class_weights_from_histogram(class_array, 'normal')


def cpu_rates(torch, cpu, mains, auxs, policy, budget_s, max_images):
    """Mpix/s of the CPU path, (a) as the reference runs it -- one image after the other, torch intra-op threads -- and (b)
    with the images spread over all host cores, each on `budget_s`/2 seconds of a bounded sample.  Returns the better one as
    the baseline, with both in the description."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    n, h, w = mains[0].shape[0], mains[0].shape[2], mains[0].shape[3]
    threads = torch.get_num_threads()
    cores = os.cpu_count() or threads

    def timed(fn):
        done, t0 = 0, time.perf_counter()
        while True:
            fn()
            done += n
            el = time.perf_counter() - t0
            if el >= budget_s / 2 or done >= max_images:
                return done, el

    cpu.step(torch, np, [m[:1] for m in mains], [a[:1] for a in auxs], policy)     # warm-up
    d_seq, t_seq = timed(lambda: cpu.step(torch, np, mains, auxs, policy))
    torch.set_num_threads(1)
    try:
        with ThreadPoolExecutor(cores) as pool:
            cpu.step(torch, np, [m[:cores] for m in mains], [a[:cores] for a in auxs], policy, pool, cores)
            d_par, t_par = timed(lambda: cpu.step(torch, np, mains, auxs, policy, pool, cores))
    finally:
        torch.set_num_threads(threads)
    mpix = h * w / 1e6
    seq, par = d_seq * mpix / t_seq, d_par * mpix / t_par
    best, used = (par, cores) if par >= seq else (seq, threads)
    sample = ("synthetic %dx%d images x 3 sources, policy '%s', %s: %d images in %.1f s as the reference's sequential loop with %d "
              "torch threads (%.2f Mpix/s), %d images in %.1f s with the images spread over %d host threads (%.2f Mpix/s); "
              "value = the better" % (w, h, policy, cpu.describe(), d_seq, t_seq, threads, seq, d_par, t_par, cores, par))
    return round(best, 3), used, sample, {"sequential_mpix_s": round(seq, 3), "image_parallel_mpix_s": round(par, 3)}


def cpu_baseline(torch, args, budget_s):
    cpu = CpuPath()
    mains, auxs = make_logits_host(torch, 16, args.height, args.width, seed=3, pin=False)
    value, used, sample, both = cpu_rates(torch, cpu, mains, auxs, args.policy, budget_s, 512)
    out = {"value": value, "unit": "Mpix/s", "cores": used, "kind": cpu.kind, "host_cpus": os.cpu_count(), "sample": sample}
    out.update(both)
    return out


def run_reference(args):
    import numpy as np
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor
    cpu = CpuPath()
    n = args.ref_images
    mains, auxs = make_logits_host(torch, n, args.height, args.width, seed=3, pin=False)
    threads, cores = torch.get_num_threads(), os.cpu_count() or 1
    # which arrangement uses this box's cores best (short probe), then W warm-up + K timed steps of that one
    _, used, probe, both = cpu_rates(torch, cpu, [m[:min(n, 8)] for m in mains], [a[:min(n, 8)] for a in auxs], args.policy, 4.0, 64)
    parallel = used == cores and cores > 1
    pool = ThreadPoolExecutor(cores) if parallel else None
    if parallel:
        torch.set_num_threads(1)

    def step():
        return cpu.step(torch, np, mains, auxs, args.policy, pool, cores) if parallel else cpu.step(torch, np, mains, auxs, args.policy)

    try:
        for _ in range(max(1, args.warmup)):
            step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            weights = step()
        el = time.perf_counter() - t0
    finally:
        if pool is not None:
            pool.shutdown()
        torch.set_num_threads(threads)
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "class_weights.npy"), weights.numpy().astype(np.float32))
    mpix = args.steps * n * args.height * args.width / 1e6
    val = round(mpix / el, 3)
    sample = ("%d synthetic %dx%d images x 3 sources per step (bounded sample of the workload), %s, %s.  Probe: %s"
              % (n, args.width, args.height, cpu.describe(),
                 "images spread over %d host threads" % cores if parallel else "sequential loop, %d torch threads" % threads, probe))
    base = {"value": val, "unit": "Mpix/s", "cores": cores if parallel else threads, "kind": cpu.kind, "sample": sample}
    base.update(both)
    emit({
        "impl": "reference", "metric": "pseudo-labelled Mpix/s (3-source fusion)", "value": val, "unit": "Mpix/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * el / args.steps, 3),
        "higher_is_better": True, "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world, *shard_plan(args, world)),
        "cpu_baseline": base,
        "e2e": {"value": val, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0})


def shard_plan(args, world):
    """(images per rank, resident pool, cycles)."""
    total = images_total(args, world)
    if total % world:
        raise SystemExit("--images-total %d does not divide over %d ranks" % (total, world))
    per_rank = total // world
    pool = per_rank if per_rank <= POOL_IMAGES else POOL_IMAGES
    if per_rank % pool:
        raise SystemExit("%d images per rank are not a whole number of %d-image pool cycles" % (per_rank, pool))
    return per_rank, pool, per_rank // pool


def workload_config(args, world, per_rank, pool, cycles):
    total = per_rank * world
    which = "configs[1]" if (world == 1 and total == 2000) else "configs[2]" if total == 20000 else "custom"
    return {"workload": "%s: 3-source fusion (camvid 13 / cityscapes 20 / forest 5 logits -> 5 greenhouse classes), class-balanced "
                        "thresholds, %d synthetic %dx%d images in all, %d per GPU" % (which, total, args.width, args.height, per_rank),
            "images_total": total, "images_per_gpu": per_rank, "resident_pool_images": pool, "pool_cycles_per_step": cycles,
            "height": args.height, "width": args.width, "policy": args.policy, "portion": args.portion,
            "sharding": "images, contiguous blocks; one all-reduce of the packed int64 statistics + three candidate-histogram all-reduces",
            "scaling_note": "N=1 is configs[1] (2,000 images); N>1 is configs[2] (20,000 images over the ranks, strong scaling); "
                            "secondary.configs2_one_gpu on the N=1 line is the same 20,000-image set on one GPU",
            "dataset": "image i of the set = image (i mod %d) of a resident pool generated from seed 3 on every rank" % pool if cycles > 1 or world > 1
                       else "resident pool generated from seed 3",
            "l2": "inputs (%.1f GB/GPU resident, every cycle reads all of it) far larger than the 126 MB L2; no flush needed"
                  % (pool * args.height * args.width * 304 / 1e9)}


_REAL_STDOUT = None


def claim_stdout():
    """Route everything libraries print on fd 1 (NCCL's version banner, torchrun notices) to stderr, so that stdout
    carries exactly ONE line: the JSON result written by emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr


def _strict(x):
    """Strict JSON has no NaN/Infinity tokens: non-finite floats become null."""
    if isinstance(x, float):
        return x if x == x and abs(x) != float("inf") else None
    if isinstance(x, dict):
        return {k: _strict(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_strict(v) for v in x]
    return x


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(_strict(line), allow_nan=False) + "\n")
    out.flush()


def full_size_checks(torch, job, pix_local, world, dist, portion, num_classes=5, ignore=4, chunk_images=500):
    """Properties that must hold for any input, verified on the very outputs of the timed run (all ranks): histograms are
    exact pixel counts, thresholding only ever moves a label to the ignore class and keeps conf >= thresh, about `portion`
    of each class survives, and the global histograms equal the sum of the per-rank bincounts.  Evaluated in slices of
    `chunk_images` images so that the temporaries stay small next to a 20,000-image shard."""
    K = num_classes
    dev = job.label.device
    local_hist = torch.zeros(K, dtype=torch.int64, device=dev)
    local_final = torch.zeros(K, dtype=torch.int64, device=dev)
    flags = {"threshold_only_moves_to_ignore": True, "kept_pixels_reach_their_threshold": True, "dropped_pixels_below_threshold": True,
             "conf_in_unit_interval": True, "uncertainty_finite_nonnegative": True}
    thresh = job.thresh
    for lo in range(0, job.label.shape[0], chunk_images):
        lab, fin, conf = job.label[lo:lo + chunk_images], job.final[lo:lo + chunk_images], job.conf[lo:lo + chunk_images]
        local_hist += torch.bincount(lab.reshape(-1).int(), minlength=K)[:K]
        local_final += torch.bincount(fin.reshape(-1).int(), minlength=K)[:K]
        changed = fin != lab
        keep = fin != ignore
        flags["threshold_only_moves_to_ignore"] &= bool((fin[changed] == ignore).all())
        flags["kept_pixels_reach_their_threshold"] &= bool((conf[keep] >= thresh[fin[keep].long()]).all())
        flags["dropped_pixels_below_threshold"] &= bool((conf[changed] < thresh[lab[changed].long()]).all())
        flags["conf_in_unit_interval"] &= bool(((conf >= 0) & (conf <= 1.0000001)).all())
        if job.unc is not None:
            unc = job.unc[lo:lo + chunk_images]
            flags["uncertainty_finite_nonnegative"] &= bool(torch.isfinite(unc).all()) and float(unc.min()) > -1e-5
    if dist is not None:
        dist.all_reduce(local_hist)
        dist.all_reduce(local_final)
    ok = {}
    ok["class_hist_is_bincount_of_labels"] = bool(torch.equal(local_hist, job.class_hist))
    ok["final_hist_is_bincount_of_final"] = bool(torch.equal(local_final, job.final_hist))
    ok["histograms_count_every_pixel"] = int(job.class_hist.sum()) == pix_local * world == int(job.final_hist.sum())
    ok["kept_equals_class_hist"] = bool(torch.equal(job.kept, job.class_hist))
    ok.update(flags)
    frac = [(int(job.final_hist[k]) / max(1, int(job.class_hist[k]))) for k in range(K) if k != ignore and int(job.class_hist[k]) > 1000]
    ok["kept_fraction_close_to_portion"] = all(abs(f - portion) < 0.01 for f in frac)
    if dist is not None:        # every rank must agree before rank 0 reports
        t = torch.tensor([int(bool(v)) for v in ok.values()], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        ok = {k: bool(f) for k, f in zip(ok, t.tolist())}
    ok["all_passed"] = all(v for v in ok.values())
    return ok


def job_digest(job):
    """sha256 over the GLOBAL results of a job (thresholds bit patterns, class / final histograms, near-tie count): equal for
    every rank count on the same image set."""
    import numpy as np
    parts = [job.thresh.detach().cpu().numpy().view(np.uint32).tobytes(), job.class_hist.cpu().numpy().tobytes(),
             job.final_hist.cpu().numpy().tobytes(), job.kept.cpu().numpy().tobytes(),
             np.int64(int(job.marginal)).tobytes()]
    return hashlib.sha256(b"".join(parts)).hexdigest()[:16]


DUMP_SAMPLE_PIXELS = 1 << 21    # 4 maps x 8 MB + 16 MB of pixel index: well under 64 MB


def dump_outputs(torch, job, out_dir, sample=DUMP_SAMPLE_PIXELS, seed=0):
    """Write the LabelJob that LabelGenerator.run returned in the last timed step to out_dir/<name>.npy, so that two builds
    can be compared output for output on the same seeded inputs.  The global thresholds and histograms are written in full;
    the per-pixel maps of this rank's shard (2.2 GB at configs[1]) at a fixed, seeded sample of `sample` flat pixel positions,
    stored beside them as `pixel_index`.  Maps and thresholds are float32, counts and the index float64 (exact).  A class that
    is never kept (the ignore class) has threshold +inf; it is written as the largest float32, which no confidence in [0, 1]
    reaches either, so that every dumped value is finite."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    npix = job.label.numel()
    idx = np.sort(np.random.default_rng(seed).choice(npix, size=min(sample, npix), replace=False))
    dev_idx = torch.from_numpy(idx).to(job.label.device)
    thresh = job.thresh.cpu().numpy().astype(np.float32)
    thresh[np.isposinf(thresh)] = np.finfo(np.float32).max
    arrays = {"pixel_index": idx.astype(np.float64), "thresh": thresh,
              "near_tie_pixels": np.array([int(job.marginal)], dtype=np.float64)}
    for name in ("label", "final", "conf", "unc"):
        arrays[name] = getattr(job, name).reshape(-1)[dev_idx].cpu().numpy().astype(np.float32)
    for name in ("kept", "class_hist", "final_hist"):
        arrays[name] = getattr(job, name).cpu().numpy().astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class Timer:
    """CUDA-event timing of `steps` calls after `warmup`, max over ranks."""

    def __init__(self, torch, dist, world, dev):
        self.torch, self.dist, self.world, self.dev = torch, dist, world, dev

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def run(self, fn, steps, warmup, finish=None):
        """finish: called after the last timed step and before the closing event (e.g. to wait for asynchronous collectives)."""
        torch = self.torch
        out = None
        for _ in range(warmup):
            out = None          # (drop the previous result first: a step may hold tens of GB of maps)
            out = fn()
        self.barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            out = None
            out = fn()
        if finish is not None:
            finish()
        t1.record()
        self.barrier()
        ms = torch.tensor([t0.elapsed_time(t1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return ms.item() / steps, out


def roofline_entry(kernel, bytes_per_launch, ms, peak, peak_src, **extra):
    achieved = bytes_per_launch / 1e9 / (ms / 1e3)
    out = {"bound": "hbm", "kernel": kernel, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
           "frac": round(achieved / peak, 4), "peak_source": peak_src, "ms_per_launch": round(ms, 4),
           "algorithmic_bytes_per_launch": int(bytes_per_launch), "traffic": None}
    out.update(extra)
    return out


# ---- secondary configurations ---------------------------------------------------------------------------------------------
def secondary_k1_policies(torch, ops, timer, mains, auxs, luts, peak, peak_src, n_img=400):
    """The per-class-probability policies of K1 ('half' = the reference's default vote, 'prob') on the first images of the
    resident pool; checked against the labels-only kernel (independent arg-max code, original class order)."""
    out = {}
    m, a = [t[:n_img] for t in mains], [t[:n_img] for t in auxs]
    n, h, w = m[0].shape[0], m[0].shape[2], m[0].shape[3]
    nbytes = n * h * w * (8 * sum(t.shape[1] for t in m) + 9)
    for policy in ("half", "prob"):
        ms, r = timer.run(lambda: ops.fuse_sources(m, a, luts, policy=policy), 5, 2)
        checks = {"conf_in_unit_interval": bool(((r.conf >= 0) & (r.conf <= 1.0000001)).all()),
                  "class_hist_is_bincount": bool(torch.equal(torch.bincount(r.label.reshape(-1).long(), minlength=5), r.class_hist))}
        if policy == "half":
            lab = ops.fuse_sources(m, a, luts, policy=policy, want_conf=False, want_unc=False, want_conf_hist=False,
                                   count_marginal=False).label
            checks["labels_equal_labels_only_kernel"] = bool(torch.equal(lab, r.label))
        checks["all_passed"] = all(checks.values())
        out["k1_policy_" + policy] = {"images": n, "mpix_per_s": round(n * h * w / 1e6 / (ms / 1e3), 1),
                                      "roofline": roofline_entry("fuse_sources_tma_kernel<GK=true> (K1, policy '%s')" % policy,
                                                                 nbytes, ms, peak, peak_src), "checks": checks}
    return out


def secondary_config0(torch, ops, timer, dev, lut20, h, w, peak, peak_src):
    """configs[0]: 1 source (20 classes, the cityscapes table), 8 images of 480x256 -- the reference's own CPU-runnable case
    (its CPU timing: BASELINE.md section 5, oracle/time_config1.py).  A launch-latency-sized job on a B200."""
    gen = torch.Generator(device=dev).manual_seed(21)
    m = torch.empty((8, 20, h, w), device=dev).normal_(0, SIGMA, generator=gen)
    a = m + torch.empty((8, 20, h, w), device=dev).normal_(0, 0.5 * SIGMA, generator=gen)
    ms, r = timer.run(lambda: ops.fuse_sources([m], [a], [lut20], policy="all"), 20, 5)
    lab = ops.fuse_sources([m], [a], [lut20], policy="all", want_conf=False, want_unc=False, want_conf_hist=False,
                           count_marginal=False).label
    z = m + 0.5 * a
    want = torch.as_tensor(lut20, device=dev)[z.argmax(1)].to(torch.uint8)         # plain torch ops on the same logits
    p = torch.softmax(z, 1)
    top2 = torch.topk(p, 2, dim=1).values
    near = (top2[:, 0] - top2[:, 1]) < 1e-6
    checks = {"labels_equal_labels_only_kernel": bool(torch.equal(lab, r.label)),
              "labels_equal_torch_argmax_table_outside_near_ties": bool(((r.label == want) | near).all()),
              # (pixels voted into the ignore class carry conf 0 by definition)
              "conf_equals_torch_softmax_max_1e-5": bool(torch.allclose(torch.where(r.label == 4, torch.zeros_like(r.conf), p.max(1).values),
                                                                        r.conf, rtol=1e-5, atol=1e-7))}
    checks["all_passed"] = all(checks.values())
    pix = 8 * h * w
    return {"configs0_one_source_8_images": {
        "ms": round(ms, 4), "mpix_per_s": round(pix / 1e6 / (ms / 1e3), 1),
        "roofline": roofline_entry("fuse_sources_tma_kernel, 1 source x 20 classes (launch-latency bound)", pix * (8 * 20 + 9), ms, peak, peak_src),
        "checks": checks}}


def secondary_loss(torch, dist, ops, timer, dev, world, rank, h, w, peak, peak_src):
    """configs[3]: uncertainty-weighted rectified CE forward + backward, B = 64 on one GPU (88 B/pixel) and the data-parallel
    share B = 8 per GPU with the global pixel count as divisor and the 3-float loss all-reduce."""
    K = 5
    gen = torch.Generator(device=dev).manual_seed(11 + rank)

    def batch(b):
        main = torch.empty((b, K, h, w), device=dev).normal_(0, SIGMA, generator=gen)
        aux = main + torch.empty((b, K, h, w), device=dev).normal_(0, 0.5 * SIGMA, generator=gen)
        target = torch.randint(1, 5, (b, h, w), device=dev, generator=gen)
        return main, aux, target

    cw = torch.tensor([1.0, 1.0, 1.0, 1.0, 0.0], device=dev)
    main, aux, target = batch(64)
    ms64, (out3, dm, da) = timer.run(lambda: ops.uw_ce_fwd_bwd(main, aux, target, cw), 10, 3)
    checks = {}
    # closed-form properties: the class gradients of every pixel sum to zero for both heads; loss = 20 * ce_part + kld_part
    scale = float(dm.abs().max())
    checks["main_gradients_sum_to_zero_per_pixel"] = float(dm.sum(1).abs().max()) <= 2e-5 * scale
    checks["aux_gradients_sum_to_zero_per_pixel"] = float(da.sum(1).abs().max()) <= 2e-5 * scale
    o = out3.tolist()
    checks["loss_is_20ce_plus_kld"] = abs(o[0] - (20.0 * o[1] + o[2])) <= 1e-5 * abs(o[0])
    # against plain PyTorch ops + autograd on a 2-image slice (the reference's expression, uest_seg_multi_os.py:1020-1023)
    m2, a2 = main[:2].clone().requires_grad_(True), aux[:2].clone().requires_grad_(True)
    p1, lp1, lp2 = torch.softmax(m2, 1), torch.log_softmax(m2, 1), torch.log_softmax(a2, 1)
    kld = (p1 * lp1 - p1 * lp2).sum(1)
    nll = -torch.log_softmax(m2 + 0.5 * a2, 1) * cw.view(1, -1, 1, 1)
    ref_loss = (nll.gather(1, target[:2].unsqueeze(1)).squeeze(1) * torch.exp(-kld)).mean() * 20 + kld.mean()
    ref_loss.backward()
    o2, dm2, da2 = ops.uw_ce_fwd_bwd(main[:2].contiguous(), aux[:2].contiguous(), target[:2].contiguous(), cw)
    g = float(m2.grad.abs().max())
    checks["loss_matches_torch_autograd_1e-5"] = abs(float(o2[0]) - float(ref_loss.detach())) <= 1e-5 * abs(float(ref_loss.detach()))
    checks["grads_match_torch_autograd_1e-4"] = bool(torch.allclose(dm2, m2.grad, rtol=1e-4, atol=1e-5 * g) and
                                                     torch.allclose(da2, a2.grad, rtol=1e-4, atol=1e-5 * g))
    del m2, a2, dm2, da2
    pix64 = 64 * h * w
    entry = {"batch": 64, "ms": round(ms64, 4), "mpix_per_s": round(pix64 / 1e6 / (ms64 / 1e3), 1),
             "roofline": roofline_entry("uw_ce_fused_kernel (K4 forward+backward, int64 targets)", pix64 * 88, ms64, peak, peak_src)}
    # data-parallel share: 8 images per GPU, divisor = global pixel count, loss parts summed over the ranks
    mb, ab, tb = main[:8].contiguous(), aux[:8].contiguous(), target[:8].contiguous()
    norm = float(world * 8 * h * w)

    def dp_step():
        o3, gm, ga = ops.uw_ce_fwd_bwd(mb, ab, tb, cw, norm_pixels=norm)
        if world > 1:
            dist.all_reduce(o3)
        return o3, gm, ga

    # The gradients need no collective (the divisor is already global); only the LOGGED loss does.  A training loop can let
    # that 12-byte all-reduce run asynchronously next to the following steps instead of in the compute stream:
    pending = []

    def dp_step_async():
        o3, gm, ga = ops.uw_ce_fwd_bwd(mb, ab, tb, cw, norm_pixels=norm)
        if world > 1:
            pending.append(dist.all_reduce(o3, async_op=True))
        return o3, gm, ga

    def drain():
        while pending:
            pending.pop().wait()

    ms8, (o3, gm, ga) = timer.run(dp_step, 20, 5)
    ms8a, _ = timer.run(dp_step_async, 20, 5, finish=drain)
    drain()
    entry["data_parallel"] = {"batch_per_gpu": 8, "global_batch": 8 * world, "ms": round(ms8, 4), "ms_loss_allreduce_async": round(ms8a, 4),
                              "mpix_per_s_all_gpus": round(world * 8 * h * w / 1e6 / (ms8 / 1e3), 1),
                              "mpix_per_s_all_gpus_async": round(world * 8 * h * w / 1e6 / (ms8a / 1e3), 1),
                              "collective": "all_reduce of 3 f32 (loss, ce part, kld part): `ms` with it in the compute stream, "
                                            "`ms_loss_allreduce_async` with async_op=True (only the logged loss needs it)" if world > 1 else "none (1 rank)",
                              "roofline": roofline_entry("uw_ce_fused_kernel, B=8 (launch-latency bound)", 8 * h * w * 88, ms8, peak, peak_src)}
    if world > 1:
        # the ranks' shares against ONE launch over the gathered global batch on every rank: same loss, and this rank's gradients
        # equal its slice of the global ones bit for bit
        gm_all = [torch.empty_like(mb) for _ in range(world)]
        ga_all = [torch.empty_like(ab) for _ in range(world)]
        gt_all = [torch.empty_like(tb) for _ in range(world)]
        dist.all_gather(gm_all, mb), dist.all_gather(ga_all, ab), dist.all_gather(gt_all, tb)
        of, gmf, gaf = ops.uw_ce_fwd_bwd(torch.cat(gm_all), torch.cat(ga_all), torch.cat(gt_all), cw)
        checks["dp_loss_equals_global_batch_loss"] = abs(float(o3[0]) - float(of[0])) <= 2e-6 * abs(float(of[0]))
        checks["dp_gradients_equal_global_batch_slice"] = bool(torch.equal(gm, gmf[8 * rank:8 * rank + 8]) and
                                                               torch.equal(ga, gaf[8 * rank:8 * rank + 8]))
    flags = torch.tensor([int(bool(v)) for v in checks.values()], device=dev)
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    checks = {k: bool(f) for k, f in zip(checks, flags.tolist())}
    checks["all_passed"] = all(checks.values())
    entry["checks"] = checks
    return {"configs3_uw_loss": entry}


def secondary_stress(torch, dist, timer, dev, world, LabelGenerator, lut20, portion, peak, peak_src):
    """configs[4]: 1024x512, three sources of 20 classes each, 256 images per GPU (a 128-image resident pool cycled twice)."""
    h, w, pool, cycles = 512, 1024, 128, 2
    src = (("a", 20), ("b", 20), ("c", 20))
    mains, auxs = make_logits_device(torch, pool, h, w, dev, seed=5, sources=src, chunk=8)
    gen = LabelGenerator([lut20] * 3, policy="all", portion=portion)
    gen.k1_events = []
    ms, job = timer.run(lambda: gen.run(mains, auxs, cycles=cycles), 5, 2)
    ev = gen.k1_events[-5 * cycles:]
    k1_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in ev) / len(ev)], device=dev)
    if world > 1:
        dist.all_reduce(k1_ms, op=dist.ReduceOp.MAX)
    pix = pool * cycles * h * w
    checks = full_size_checks(torch, job, pix, world, dist if world > 1 else None, portion)
    entry = {"workload": "1024x512, 3 sources x 20 classes (cityscapes table), %d images per GPU = %d-image pool x %d cycles, thresholds"
                         % (pool * cycles, pool, cycles),
             "ms_per_step": round(ms, 4), "mpix_per_s_all_gpus": round(world * pix / 1e6 / (ms / 1e3), 1),
             "whole_step_frac_495B_per_pix": round(pix * 495 / 1e9 / (ms / 1e3) / peak, 4),
             "roofline": roofline_entry("fuse_sources_tma_kernel (K1), 489 B/pixel", pool * h * w * 489, k1_ms.item(), peak, peak_src),
             "checks": checks, "digest": job_digest(job)}
    del mains, auxs, job
    torch.cuda.empty_cache()
    return {"configs4_stress_1024x512": entry}


def secondary_lowres(torch, ops, timer, dev, luts, h, w, peak, peak_src, n_img=200):
    """(f)1: K1 with the networks' closing bilinear upsample fused in (main head at H/2 x W/2, aux head at H/4 x W/4)."""
    import torch.nn.functional as F
    mains, auxs = make_logits_device(torch, n_img, h, w, dev, seed=9, lowres=True)
    ms, r = timer.run(lambda: ops.fuse_sources_lowres(mains, auxs, luts, (h, w), policy="all"), 5, 2)
    # against upsample-then-fuse on a few images: the kernel and ATen round the interpolated logit differently in the last
    # place, so labels may differ at near-ties only and confidences agree to 1e-4
    k = 4
    up = lambda t: F.interpolate(t[:k], size=(h, w), mode="bilinear", align_corners=True).contiguous()
    full = ops.fuse_sources([up(t) for t in mains], [up(t) for t in auxs], luts, policy="all")
    diff = (full.label != r.label[:k])
    same = ~diff
    checks = {"label_mismatch_fraction_below_1e-3": float(diff.float().mean()) < 1e-3,
              "conf_within_1e-4_where_labels_agree": bool(torch.allclose(r.conf[:k][same], full.conf[same], rtol=1e-4, atol=1e-6)),
              "unc_within_1e-4": bool(torch.allclose(r.unc[:k], full.unc, rtol=1e-4, atol=5e-6))}
    checks["all_passed"] = all(checks.values())
    pix = n_img * h * w
    nbytes = pix * (4 * sum(t.shape[1] for t in mains) * (1 / 4 + 1 / 16) + 9)
    entry = {"images": n_img, "gpix_per_s": round(pix / 1e9 / (ms / 1e3), 2), "ms": round(ms, 4),
             "roofline": roofline_entry("fuse_sources_lowres_kernel (instruction-bound; 56.5 B/pixel)", nbytes, ms, peak, peak_src),
             "checks": checks}
    del mains, auxs
    torch.cuda.empty_cache()
    return {"k1_lowres_fused_upsample": entry}


def h2d_ceiling(torch, timer, dev, tensors):
    """Bare pinned host -> device copy of the same buffers, all ranks at once: GB/s of this rank (min over ranks reported)."""
    dst = [torch.empty_like(t, device=dev) for t in tensors]
    nbytes = sum(t.numel() * 4 for t in tensors)

    def copy_all():
        for d, s in zip(dst, tensors):
            d.copy_(s, non_blocking=True)

    ms, _ = timer.run(copy_all, 3, 1)
    return nbytes / 1e9 / (ms / 1e3)


def main():
    args = parse_args()
    claim_stdout()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import torch.distributed as dist
    from mspl_b200 import _lib, ops
    from mspl_b200.data_loader.segmentation.greenhouse import SOURCE_TABLES
    from mspl_b200.pipeline import LabelGenerator

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    sampler = ClockSampler(local, int(os.environ.get("MSPL_BENCH_CLOCK_PERIOD_MS", "20")))
    if rank == 0:
        sampler.start()
    timer = Timer(torch, dist, world, dev)
    h, w = args.height, args.width
    per_rank, pool, cycles = shard_plan(args, world)
    pix_local = per_rank * h * w
    luts = [SOURCE_TABLES[s] for s, _ in SOURCES]
    peak, peak_src = hbm_peak()
    mains, auxs = make_logits_device(torch, pool, h, w, dev, seed=3)
    gen = LabelGenerator(luts, policy=args.policy, portion=args.portion)
    torch.cuda.synchronize()

    # ---- the timed steps ---------------------------------------------------------------------------------------------
    job = None
    for _ in range(args.warmup):
        job = None
        job = gen.run(mains, auxs, cycles=cycles)
    timer.barrier()
    gen.k1_events = []      # CUDA events around every K1 launch (roofline of the dominant kernel, measured live)
    launches0, coll0 = gen.launches, gen.collectives
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.time()
    t0.record()
    for _ in range(args.steps):
        job = None              # the previous step's maps go back to the caching allocator before the next step takes its own
        job = gen.run(mains, auxs, cycles=cycles)
    t1.record()
    timer.barrier()
    wall1 = time.time()
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
    k1_events = list(gen.k1_events)
    gen.k1_events = None
    k1_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in k1_events) / max(1, len(k1_events))], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(k1_ms, op=dist.ReduceOp.MAX)
    ms_per_step = ms.item() / args.steps
    launches = gen.launches - launches0
    collectives = (gen.collectives - coll0) / max(1, args.steps)
    value = world * pix_local / 1e6 / (ms_per_step / 1e3)

    # ---- roofline of the dominant kernel (K1): algorithmic bytes = 8*sum(C_s) + 9 per pixel (SURVEY.md 8d) ----
    k1_bytes = pool * h * w * (8 * sum(c for _, c in SOURCES) + 9)
    traffic = ncu_traffic()
    roofline = roofline_entry("fuse_sources_tma_kernel (K1)", k1_bytes, k1_ms.item(), peak, peak_src)
    per_launch_scale = k1_bytes / traffic["algorithmic_bytes_at_capture"] if traffic and traffic.get("algorithmic_bytes_at_capture") else None
    roofline.update({
        "traffic": int(traffic["bytes_per_launch"] * per_launch_scale) if per_launch_scale else None,
        "traffic_note": traffic.get("note") if traffic else "no ncu capture committed yet",
        "launches_per_step": cycles,
        "share_of_step": round(k1_ms.item() * cycles / ms_per_step, 4),
        "whole_step_frac_319B_per_pix": round(pix_local * 319 / 1e9 / (ms_per_step / 1e3) / peak, 4),
        "variant": lib.mspl_fuse_variant().decode()})

    # ---- size-independent properties at the full benchmark size (the CPU oracle cannot run thousands of images) -----------
    checks = full_size_checks(torch, job, pix_local, world, dist if world > 1 else None, args.portion)
    results = {"near_tie_pixels": int(job.marginal.item()), "class_hist": job.class_hist.tolist(), "final_hist": job.final_hist.tolist(),
               # the never-selected ignore class has threshold +inf: emit() writes it as null (strict JSON has no Infinity)
               "thresholds": [round(x, 6) for x in job.thresh.tolist()], "kept": job.kept.tolist(),
               "digest": job_digest(job),
               "digest_note": "sha256/16 of (thresholds, class_hist, final_hist, kept, near-tie count): identical for every rank "
                              "count on the same image set (compare configs[2] lines and secondary.configs2_one_gpu)"}
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, job, args.dump_outputs)
    job = None

    # ---- end to end through the public host-buffer API -----------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        ne = min(args.e2e_images, pool)
        hm, ha = make_logits_host(torch, ne, h, w, seed=7 + rank, pin=True)
        out_host = torch.empty((ne, h, w), dtype=torch.uint8, pin_memory=True)
        ems_step, _ = timer.run(lambda: gen.run_from_host(hm, ha, dev, out_host=out_host), args.e2e_steps, 1)
        in_bytes = ne * h * w * 8 * sum(c for _, c in SOURCES)
        ceil_gbs = torch.tensor([h2d_ceiling(torch, timer, dev, hm + ha)], device=dev)
        if world > 1:
            dist.all_reduce(ceil_gbs, op=dist.ReduceOp.MIN)
        got_gbs = in_bytes / 1e9 / (ems_step / 1e3)
        e2e = {"value": round(world * ne * h * w / 1e6 / (ems_step / 1e3), 1), "unit": "Mpix/s",
               "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": ne * h * w,
               "images_per_step_per_gpu": ne, "ms_per_step": round(ems_step, 3),
               "h2d_gbs_per_gpu": round(got_gbs, 2), "h2d_ceiling_gbs": round(ceil_gbs.item(), 2),
               "frac_of_ceiling": round(got_gbs / ceil_gbs.item(), 4),
               "ceiling_note": "bare pinned copy_ of the same buffers, all %d ranks copying at once, slowest rank" % world,
               "api": "mspl_b200.pipeline.LabelGenerator.run_from_host (pinned host logits -> uint8 label maps on host)"}
        del hm, ha
        # the same job through the (f)1 boundary: the sources hand over their heads BEFORE the closing upsample (47.5 B/pixel in)
        hm, ha = make_logits_host(torch, ne, h, w, seed=7 + rank, pin=True, lowres=True)
        lms_step, _ = timer.run(lambda: gen.run_from_host(hm, ha, dev, out_host=out_host, out_size=(h, w)), args.e2e_steps, 1)
        lr_bytes = sum(t.numel() * 4 for t in hm + ha)
        e2e["fused_upsample_boundary"] = {
            "value": round(world * ne * h * w / 1e6 / (lms_step / 1e3), 1), "unit": "Mpix/s", "h2d_bytes_per_step": lr_bytes,
            "d2h_bytes_per_step": ne * h * w, "ms_per_step": round(lms_step, 3),
            "note": "NOT the headline: same images through LabelGenerator.run_from_host(out_size=...), inputs = pre-upsample heads "
                    "(main H/2 x W/2, aux H/4 x W/4), interpolation inside K1-lowres"}
        del hm, ha

    # ---- secondary configurations (each frees what it allocates; the main pool goes first where memory is needed) ----------
    secondary = {}
    if not args.no_secondary:
        secondary.update(secondary_k1_policies(torch, ops, timer, mains, auxs, luts, peak, peak_src))
        if world == 1 and per_rank * world != 20000:
            mains = auxs = None
            torch.cuda.empty_cache()
            mains, auxs = make_logits_device(torch, POOL_IMAGES, h, w, dev, seed=3)
            c2 = 20000 // POOL_IMAGES
            g2 = LabelGenerator(luts, policy=args.policy, portion=args.portion)
            ms2, job2 = timer.run(lambda: g2.run(mains, auxs, cycles=c2), 3, 1)
            pix2 = 20000 * h * w
            secondary["configs2_one_gpu"] = {
                "workload": "configs[2]'s 20,000-image set on ONE GPU: %d cycles over the resident %d-image pool" % (c2, POOL_IMAGES),
                "ms_per_step": round(ms2, 3), "mpix_per_s": round(pix2 / 1e6 / (ms2 / 1e3), 1),
                "whole_step_frac_319B_per_pix": round(pix2 * 319 / 1e9 / (ms2 / 1e3) / peak, 4),
                "checks": full_size_checks(torch, job2, pix2, 1, None, args.portion), "digest": job_digest(job2)}
            job2 = None
        mains = auxs = None
        torch.cuda.empty_cache()
        secondary.update(secondary_config0(torch, ops, timer, dev, SOURCE_TABLES["cityscapes"], h, w, peak, peak_src))
        secondary.update(secondary_loss(torch, dist, ops, timer, dev, world, rank, h, w, peak, peak_src))
        secondary.update(secondary_stress(torch, dist, timer, dev, world, LabelGenerator, SOURCE_TABLES["cityscapes"], args.portion,
                                          peak, peak_src))
        secondary.update(secondary_lowres(torch, ops, timer, dev, luts, h, w, peak, peak_src))

    if rank == 0:
        cpu = None if args.no_cpu else cpu_baseline(torch, args, args.cpu_seconds)
        line = {
            "metric": "pseudo-labelled Mpix/s (3-source fusion)", "value": round(value, 1), "unit": "Mpix/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
            "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world, per_rank, pool, cycles),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
            "collectives_per_step": collectives, "clocks": clocks, "checks": checks, "results": results, "secondary": secondary,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
