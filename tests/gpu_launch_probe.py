"""Helpers shared by the -m gpu files that check persistent-kernel paths against the oracle: record which kernels a call
launched (torch.profiler), assert the instantiation and that its grid loops over more than one pass, and compare a K1
result with the oracle.  Test infrastructure only."""
import contextlib
import json
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle import mspl_oracle as O

RTOL = 1e-5
KLD_ATOL = 2e-6

Launch = namedtuple("Launch", "name grid smem")      # name without spaces, CTAs launched, shared memory per CTA (bytes)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ops():
    from mspl_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def sms(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


@pytest.fixture
def launches(tmp_path):
    """launches(fn) runs fn() under torch.profiler (CUDA activity only) and returns (fn's result, [Launch] of every kernel)."""
    count = [0]

    def run(fn):
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        count[0] += 1
        path = tmp_path / ("trace%d.json" % count[0])
        prof.export_chrome_trace(str(path))
        with open(path) as f:
            events = json.load(f)["traceEvents"]
        ks = [Launch(e["name"].replace(" ", ""), int(np.prod(e["args"]["grid"])), int(e["args"]["shared memory"]))
              for e in events if e.get("cat") == "kernel"]
        assert ks, "torch.profiler recorded no CUDA kernel: cannot tell which instantiation ran"
        return out, ks
    return run


def _the(ks, fragment):
    """The one launch whose demangled name (spaces removed) contains `fragment`."""
    hits = [k for k in ks if fragment in k.name]
    assert len(hits) == 1, "expected one launch of %s, got %d; kernels: %s" % (fragment, len(hits), sorted({k.name[:90] for k in ks}))
    return hits[0]


def _repeats(k, work, per_cta_pass=1):
    """The launch's CTAs cover `work` units (tiles, or pixel groups at per_cta_pass per CTA and pass) in more than one pass."""
    assert work > k.grid * per_cta_pass, "%s: %d units fit into one pass of %d CTAs" % (k.name[:60], work, k.grid)


@contextlib.contextmanager
def _oracle_settings(ignore=4, margin=None):
    """O.merge_outputs writes the reference's hard-coded ignore id; the fused-upsample definition widens the near-tie margin."""
    saved = O.IGNORE_LABEL, O.NEAR_TIE_MARGIN
    O.IGNORE_LABEL = ignore
    if margin is not None:
        O.NEAR_TIE_MARGIN = margin
    try:
        yield
    finally:
        O.IGNORE_LABEL, O.NEAR_TIE_MARGIN = saved


def _check_fusion(ops, r, ref, K, ignore, conf_rtol=RTOL, conf_atol=1e-7, unc_rtol=RTOL, unc_atol=KLD_ATOL, ds_rate=1):
    """Labels except at counted near-ties, conf / unc, the class histogram (== the label map's, == the oracle's when every
    label agrees), the fused confidence histogram (the pixels with (row*W + col) % ds_rate == 0), and select_and_apply on it
    against the sort definition."""
    lab, conf = r.label.cpu(), r.conf.cpu()
    diff = lab != ref["label"]
    assert not bool((diff & ~ref["marginal"]).any()), "%d mismatches outside near-ties" % int((diff & ~ref["marginal"]).sum())
    torch.testing.assert_close(conf[~diff], ref["conf"][~diff], rtol=conf_rtol, atol=conf_atol)
    torch.testing.assert_close(r.unc.cpu(), ref["unc"], rtol=unc_rtol, atol=unc_atol)
    assert torch.equal(r.class_hist.cpu(), torch.bincount(lab.reshape(-1).long(), minlength=K))
    if not bool(diff.any()):
        assert torch.equal(r.class_hist.cpu(), ref["class_hist"])
    h, w = lab.shape[-2:]
    keep = (torch.arange(h * w) % ds_rate == 0).reshape(h, w).expand(lab.shape)
    assert torch.equal(r.conf_hist.sum(dim=1).cpu(), torch.bincount(lab[keep].long(), minlength=K))
    th_ref, kept_ref = O.cb_thresholds(lab, conf, 0.2, ds_rate, K, ignore=ignore)
    f_ref, m_ref = O.apply_thresholds(lab, conf, th_ref, ignore)
    th, kept, final, mask, fh = ops.select_and_apply(r.label, r.conf, 0.2, ds_rate, K, ignore, conf_hist=r.conf_hist.clone(),
                                                     want_mask=True)
    assert torch.equal(th.cpu(), th_ref) and torch.equal(kept.cpu(), kept_ref)
    assert torch.equal(final.cpu(), f_ref) and torch.equal(mask.cpu(), m_ref)
    assert torch.equal(fh.cpu(), torch.bincount(f_ref.reshape(-1).long(), minlength=K))
