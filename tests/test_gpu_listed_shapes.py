"""-m gpu: the greenhouse tables' sources run K1's straight-line bodies (compiled chunk shapes, kSourceShapes in pixel_math.cuh:
group commits only at group ends, no first-chunk rescale, no padded tail classes), and those give, pixel for pixel, the same
bits as the scalar fallback kernel, which pads tail chunks and rescales every chunk.

The fallback is forced by a width that breaks H*W % 4: its input holds the TMA input's pixels plus one extra column, so the
pixels shared by both runs carry the same logits, and every per-pixel output (label, confidence, uncertainty, each source's
KLD) must be bit-equal there.  The 4-source set has 11 chunks per tile, so consecutive tiles of a CTA start on different ring
stages; the 255-row image ends in a partial tile."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import mspl_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gpu_launch_probe import _repeats, _the, dev, launches, ops, sms  # noqa: E402,F401

pytestmark = pytest.mark.gpu

TILE = 960


def _shape_ids(names):
    import ctypes
    from mspl_b200 import _lib
    lib = _lib.load()
    out = []
    for nm in names:
        lut = np.asarray(O.LUTS[nm])
        out.append(lib.mspl_class_order_shape((ctypes.c_ubyte * len(lut))(*[int(v) for v in lut]), len(lut), 5))
    return out


@pytest.mark.parametrize("K", [5, 8])
@pytest.mark.parametrize("sigma", [3.0, 40.0])
@pytest.mark.parametrize("names", [("camvid", "cityscapes", "forest"), ("camvid", "cityscapes", "forest", "camvid")])
def test_listed_shapes_match_the_scalar_kernel(ops, dev, sms, launches, names, sigma, K):
    assert all(_shape_ids(names)), "the shipped tables must have compiled shapes"
    n, h, w = 4, 255, 480
    assert (h * (w + 1)) % 4 != 0
    n_tiles = n * -(-(h * w) // TILE)
    mains, auxs = [], []
    for i, nm in enumerate(names):
        m, a = O.synthetic_logits(n, len(O.LUTS[nm]), h, w + 1, seed=500 + 10 * i + int(sigma), sigma=sigma)
        mains.append(m.to(dev)), auxs.append(a.to(dev))
    tma_m = [m[..., :w].contiguous() for m in mains]
    tma_a = [a[..., :w].contiguous() for a in auxs]
    luts = [O.LUTS[nm] for nm in names]
    S = len(names)
    ignore = 4 if K == 5 else 6
    KT, nst = (5, 4) if K == 5 else (8, 3)
    for policy in ("all", "half", "prob"):
        gk = policy == "prob" or ops.vote_threshold(S, policy) < S
        kw = dict(policy=policy, num_classes=K, ignore_label=ignore, want_kld=True)
        r, ks = launches(lambda: ops.fuse_sources(tma_m, tma_a, luts, **kw))
        _repeats(_the(ks, "fuse_sources_tma_kernel<15,2,5,%d,%d,%s>" % (nst, KT, str(gk).lower())), n_tiles)
        s, ks = launches(lambda: ops.fuse_sources(mains, auxs, luts, **kw))
        _the(ks, "fuse_sources_direct_kernel<5,%d,%s," % (KT, str(gk).lower()))
        assert torch.equal(r.label, s.label[..., :w]), policy
        assert torch.equal(r.conf, s.conf[..., :w]), policy
        assert torch.equal(r.unc, s.unc[..., :w]), policy
        for a, b in zip(r.kld, s.kld):
            assert torch.equal(a, b[..., :w]), policy
        assert torch.equal(r.class_hist.cpu(), torch.bincount(r.label.reshape(-1).long().cpu(), minlength=K))
