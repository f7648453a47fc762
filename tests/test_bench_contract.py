"""CPU tests of bench.py's host logic: the reference arm prints exactly one strict-JSON line with the contract's keys, the
image-parallel arrangement of the CPU port computes the same labels and class counts as the sequential loop, and non-finite
floats never reach the output."""
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import mspl_oracle as O  # noqa: E402


def test_strict_json_has_no_nan_or_infinity():
    line = {"a": [1.0, float("inf"), float("-inf"), float("nan")], "b": {"c": (2, 3.5, float("inf"))}, "d": "inf", "e": None}
    out = json.dumps(bench._strict(line), allow_nan=False)
    assert json.loads(out) == {"a": [1.0, None, None, None], "b": {"c": [2, 3.5, None]}, "d": "inf", "e": None}


def test_image_parallel_arrangement_equals_sequential_loop():
    """Both arrangements of the CPU arm (the reference's sequential loop; images dealt to worker threads) give the same class
    weights, with the live reference's functions (when /root/reference or oracle/_ref is present) and with the oracle port."""
    mains, auxs = bench.make_logits_host(torch, 5, 24, 32, seed=3, pin=False)
    cpu = bench.CpuPath()
    for policy in ("all", "half"):
        w_seq = cpu.step(torch, np, mains, auxs, policy)
        with ThreadPoolExecutor(3) as pool:
            w_par = cpu.step(torch, np, mains, auxs, policy, pool, 3)
        assert torch.equal(w_seq, w_par)
        _, class_array = O.multi_source_labels(mains, auxs, [O.LUTS[s] for s, _ in bench.SOURCES], policy)
        assert torch.equal(w_seq, O.class_weights_from_histogram(class_array, 'normal'))     # reference arm == oracle port


def test_shard_plan_covers_the_named_configs():
    import argparse
    a = argparse.Namespace(images_total=0)
    assert bench.shard_plan(a, 1) == (2000, 2000, 1)              # configs[1]
    assert bench.shard_plan(a, 2) == (10000, 2500, 4)             # configs[2]: 20,000 images over the ranks
    assert bench.shard_plan(a, 4) == (5000, 2500, 2)
    assert bench.shard_plan(a, 8) == (2500, 2500, 1)
    a.images_total = 20000
    assert bench.shard_plan(a, 1) == (20000, 2500, 8)


def test_dump_outputs_writes_the_job_as_float_arrays(tmp_path):
    """--dump-outputs: every array of the LabelJob as float32/float64 .npy, the maps at a seeded pixel sample that is the same
    on every call, and the whole dump under 64 MB at the size of configs[1]."""
    from mspl_b200.pipeline import LabelJob
    n, h, w = 3, 16, 20
    gen = torch.Generator().manual_seed(1)
    label = torch.randint(0, 5, (n, h, w), generator=gen).to(torch.uint8)
    final = torch.where(torch.rand(n, h, w, generator=gen) < 0.2, torch.full_like(label, 4), label)
    conf, unc = torch.rand(n, h, w, generator=gen), torch.rand(n, h, w, generator=gen)
    hist = torch.bincount(label.reshape(-1).long(), minlength=5)
    job = LabelJob(label, final, None, conf, unc, torch.tensor([0.5, 0.25, 0.75, 0.125, float("inf")]), hist, hist,
                   torch.bincount(final.reshape(-1).long(), minlength=5), torch.tensor(7))
    for d in ("a", "b"):
        bench.dump_outputs(torch, job, str(tmp_path / d), sample=100)
    names = {"pixel_index", "label", "final", "conf", "unc", "thresh", "kept", "class_hist", "final_hist", "near_tie_pixels"}
    assert {f[:-4] for f in os.listdir(tmp_path / "a")} == names
    for name in names:
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.dtype in (np.float32, np.float64) and np.isfinite(a).all() and np.array_equal(a, b), name
    # the never-kept ignore class: +inf becomes the largest float32, the other thresholds are written as they are
    assert np.load(tmp_path / "a" / "thresh.npy").tolist() == [0.5, 0.25, 0.75, 0.125, float(np.finfo(np.float32).max)]
    idx = np.load(tmp_path / "a" / "pixel_index.npy").astype(np.int64)
    assert len(idx) == 100 and len(np.unique(idx)) == 100 and idx.max() < n * h * w
    for name, t in (("label", label), ("final", final), ("conf", conf), ("unc", unc)):
        assert np.array_equal(np.load(tmp_path / "a" / (name + ".npy")), t.reshape(-1).numpy()[idx].astype(np.float32)), name
    assert np.array_equal(np.load(tmp_path / "a" / "final_hist.npy"), job.final_hist.numpy().astype(np.float64))
    assert np.load(tmp_path / "a" / "near_tie_pixels.npy").tolist() == [7.0]
    assert bench.DUMP_SAMPLE_PIXELS < 2000 * 256 * 480
    assert 4 * 4 * bench.DUMP_SAMPLE_PIXELS + 8 * bench.DUMP_SAMPLE_PIXELS <= 64 << 20     # 4 float32 maps + float64 index


def test_reference_arm_prints_one_contract_line(tmp_path):
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                        "--warmup", "1", "--ref-images", "2", "--height", "32", "--width", "48", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, env=env, timeout=600)
    # --dump-outputs: the class weights of the last timed step, as the oracle port computes them on the same seeded inputs
    mains, auxs = bench.make_logits_host(torch, 2, 32, 48, seed=3, pin=False)
    _, class_array = O.multi_source_labels(mains, auxs, [O.LUTS[s] for s, _ in bench.SOURCES], "all")
    assert os.listdir(tmp_path) == ["class_weights.npy"], p.stderr[-2000:]
    got = np.load(tmp_path / "class_weights.npy")
    assert got.dtype == np.float32 and np.array_equal(got, O.class_weights_from_histogram(class_array, 'normal').numpy())
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0], parse_constant=lambda c: (_ for _ in ()).throw(ValueError("non-strict JSON constant " + c)))
    assert d["impl"] == "reference" and d["unit"] == "Mpix/s" and d["higher_is_better"] is True
    assert d["metric"] == "pseudo-labelled Mpix/s (3-source fusion)" and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1 and d["gpu_launches"] == 0
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_silently():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1", PYTHONDONTWRITEBYTECODE="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, env=env, timeout=600)
    assert p.returncode == 0 and p.stdout.strip() == ""
