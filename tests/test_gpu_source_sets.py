"""-m gpu: K1 and K1-lowres on source sets beyond the three-source (13 / 20 / 5 classes) set of the other at-scale cases --
4 and 8 sources, 256-class and 1-class sources, sources with different head sizes in K1-lowres -- and the hard-label vote
kernel at up to 15 sources, against the CPU oracle with the tolerances of tests/test_gpu_parity.py.

Every fused case runs over enough tiles that each persistent CTA runs several, and its class counts are chosen so that the
number of class chunks per tile (sum over sources of ceil(C_s / 5)) is not a multiple of the ring's stage count: consecutive
tiles of a CTA start on different ring stages and mbarrier phases.  The test asserts that arithmetic, and from the profiler
which instantiation ran and that its grid loops over more than one pass.

The oracle runs each source alone (O.fuse_sources with one source) and _combine forms O.fuse_sources' closing sums for every
policy from those per-source results; test_k1_many_sources checks that this equals O.fuse_sources on the first image."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import mspl_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gpu_launch_probe import (KLD_ATOL, RTOL, _check_fusion, _oracle_settings, _repeats, _the,  # noqa: E402,F401
                              dev, launches, ops, sms)

pytestmark = pytest.mark.gpu

CH = 5                              # kFuseChunk: source classes per ring stage
TILE = 960                          # pixels per tile of the TMA and lowres kernels (15 consumer warps x 32 lanes x 2 pixels)
LEAN = dict(want_conf=False, want_unc=False, want_conf_hist=False, count_marginal=False)     # -> the labels-only kernel
LOWRES_TOL = dict(conf_rtol=1e-4, conf_atol=1e-6, unc_rtol=1e-4, unc_atol=1e-5)             # test_fuse_sources_lowres's parity


def _ignore(K):
    return 4 if K == 5 else 6


def _ring_carry(classes, nstage):
    """A tile's chunks do not fill a whole number of ring cycles, so the next tile of the CTA starts mid-ring."""
    chunks = sum(-(-c // CH) for c in classes)
    assert chunks % nstage != 0, "%d chunks per tile: every tile starts on ring stage 0" % chunks


def _tables(classes, K, ignore, gen):
    """Random tables onto [0, K); source 0 never maps to target 1, source 1 maps its first class onto the ignore class."""
    luts = [torch.randint(0, K, (c,), generator=gen).numpy() for c in classes]
    luts[0][luts[0] == 1] = 2
    luts[1][0] = ignore
    assert 1 not in luts[0] and ignore in luts[1]
    return luts


def _per_source_oracle(mains, auxs, luts, K, ignore):
    """O.fuse_sources of each source alone: its labels (one source, 'all': the table lookup itself), G_s ('fused'), D_s ('unc')
    and near-tie flags.  Run under the caller's _oracle_settings."""
    return [O.fuse_sources([m], [a], [lut], "all", K, ignore) for m, a, lut in zip(mains, auxs, luts)]


def _combine(per, policy, K, ignore):
    """O.fuse_sources' closing steps for `policy` on per-source results: fp32 sums in source order, then the vote or the
    probability argmax.  Run under the same _oracle_settings as _per_source_oracle."""
    S = len(per)
    fsum, usum = torch.zeros_like(per[0]["fused"]), torch.zeros_like(per[0]["unc"])
    marginal = torch.zeros_like(per[0]["marginal"])
    for r in per:
        fsum, usum = fsum + r["fused"], usum + r["unc"]
        marginal = marginal | r["marginal"]
    fm, unc = fsum / S, usum / S
    if policy == "prob":
        label = torch.from_numpy(np.argmax(fm.numpy(), axis=1))
        conf = fm.max(dim=1).values
        t2 = torch.topk(fm, 2, dim=1).values
        marginal = marginal | ((t2[:, 0] - t2[:, 1]) < O.NEAR_TIE_MARGIN)
    else:
        stack = torch.stack([r["label"] for r in per]).numpy()
        label = torch.from_numpy(np.stack([O.merge_outputs(stack[:, i], K, policy) for i in range(stack.shape[1])]))
        conf = torch.gather(fm, 1, label.unsqueeze(1)).squeeze(1)
        conf = torch.where(label == ignore, torch.zeros_like(conf), conf)
    return dict(label=label.to(torch.uint8), conf=conf, unc=unc, kld=[r["kld"][0] for r in per],
                class_hist=torch.bincount(label.reshape(-1), minlength=K)[:K], marginal=marginal)


def _assert_combine_is_the_oracle(mains, auxs, luts, K, ignore, policies):
    one = ([m[:1] for m in mains], [a[:1] for a in auxs])
    with _oracle_settings(ignore):
        per = _per_source_oracle(*one, luts, K, ignore)
        for policy in policies:
            got, want = _combine(per, policy, K, ignore), O.fuse_sources(*one, luts, policy, K, ignore)
            for key in ("label", "conf", "unc", "class_hist", "marginal"):
                assert torch.equal(got[key], want[key]), (policy, key)


def _exact_target_ties(mains, auxs, luts, K):
    """Pixels where, for some source, the best z of two different targets is exactly equal (z = main + 0.5 aux)."""
    tie = torch.zeros(mains[0].shape[0], *mains[0].shape[2:], dtype=torch.bool)
    for m, a, lut in zip(mains, auxs, luts):
        z = m + 0.5 * a
        lut_t = torch.as_tensor(lut)
        present = [k for k in range(K) if bool((lut_t == k).any())]
        if len(present) > 1:
            top2 = torch.topk(torch.stack([z[:, lut_t == k].max(dim=1).values for k in present], dim=1), 2, dim=1).values
            tie |= top2[:, 0] == top2[:, 1]
    return tie


def _offset_views(ts, dev):
    """Copies of `ts` that start 4 bytes past a 16-byte boundary: the scalar (direct) kernel instead of the TMA one."""
    out = []
    for t in ts:
        buf = torch.empty(t.numel() + 1, device=dev)
        buf[1:] = t.reshape(-1)
        out.append(buf[1:].view(t.shape))
    return out


# ---- 1. K1 with 4 and 8 sources over many tiles per CTA -------------------------------------------------------------------
SOURCE_SETS = {"s8": (2, 3, 5, 7, 11, 13, 17, 19),      # 19 chunks per tile: 3 mod 4, 1 mod 3
               "s4": (13, 20, 5, 7)}                      # 10 chunks: 2 mod 4, 1 mod 3


@pytest.mark.parametrize("K", [5, 8])
@pytest.mark.parametrize("name", ["s8", "s4"])
def test_k1_many_sources(ops, dev, sms, launches, name, K):
    """8 x 256x480 (1,024 tiles, about seven per CTA), random tables onto K = 5 / 8, every policy kind: 'half', 'all', S
    (no per-target maxima), S - 1 and 1 (with them), 0 (clamped to 1: nothing can become the ignore class), 'prob'.  All S
    per-source KLD maps; 'half' with ds_rate = 3 into select_and_apply; the labels-only kernel under every vote policy; the
    scalar kernel on 4-byte-offset views bit for bit against the TMA kernel.  The 8-source set has quantised logits (z exact,
    many exact ties between targets): under vote policies its labels must match the oracle bit for bit, with no near-tie
    excused, and the oracle may flag a near-tie only where two targets tie exactly."""
    classes = SOURCE_SETS[name]
    S, n, h, w = len(classes), 8, 256, 480
    ignore, KT, nst = _ignore(K), (5 if K == 5 else 8), (4 if K == 5 else 3)
    n_tiles = n * -(-(h * w) // TILE)
    assert n_tiles >= 6 * sms
    _ring_carry(classes, nst)
    quantised = name == "s8"
    gen = torch.Generator().manual_seed(100 * S + K)
    mains, auxs = [], []
    for s, c in enumerate(classes):
        m, a = O.synthetic_logits(n, c, h, w, seed=1000 * S + 10 * K + s)
        if quantised:
            m, a = torch.round(m), torch.round(2 * a) / 2
        mains.append(m), auxs.append(a)
    luts = _tables(classes, K, ignore, gen)
    policies = ("half", "all", S, S - 1, 1, 0, "prob")
    _assert_combine_is_the_oracle(mains, auxs, luts, K, ignore, ("half", S - 1, "prob"))
    with _oracle_settings(ignore):
        per = _per_source_oracle(mains, auxs, luts, K, ignore)
    ties = _exact_target_ties(mains, auxs, luts, K) if quantised else None
    md, ad = [m.to(dev) for m in mains], [a.to(dev) for a in auxs]
    offs = _offset_views(md + ad, dev)
    labels_at = {}
    for policy in policies:
        with _oracle_settings(ignore):
            ref = _combine(per, policy, K, ignore)
        gk = policy == "prob" or max(ops.vote_threshold(S, policy), 1) < S
        ds = 3 if policy == "half" else 1
        kw = dict(policy=policy, num_classes=K, ignore_label=ignore, ds_rate=ds)
        r, ks = launches(lambda: ops.fuse_sources(md, ad, luts, want_kld=True, **kw))
        _repeats(_the(ks, "fuse_sources_tma_kernel<15,2,5,%d,%d,%s>" % (nst, KT, str(gk).lower())), n_tiles)
        _check_fusion(ops, r, ref, K, ignore, ds_rate=ds)
        for got, want in zip(r.kld, ref["kld"]):        # one source's KLD: absolute floor x sigma, as in test_gpu_fuzz.py
            torch.testing.assert_close(got.cpu(), want, rtol=RTOL, atol=3 * KLD_ATOL)
        labels_at[policy] = r.label
        if policy != "prob":
            if quantised:
                assert torch.equal(r.label.cpu(), ref["label"])
                assert not bool((ref["marginal"] & ~ties).any()), "near-ties flagged where no two targets tie exactly"
            lean, ks = launches(lambda: ops.fuse_sources(md, ad, luts, policy=policy, num_classes=K, ignore_label=ignore, **LEAN))
            _repeats(_the(ks, "fuse_labels_tma_kernel<15,2,5,%d,%d>" % (nst, KT)), n_tiles)
            assert torch.equal(lean.label, r.label) and torch.equal(lean.class_hist, r.class_hist)
        s, ks = launches(lambda: ops.fuse_sources(offs[:S], offs[S:], luts, **kw))
        _repeats(_the(ks, "fuse_sources_direct_kernel<5,%d,%s," % (KT, str(gk).lower())), n * h * w, 256)
        assert torch.equal(s.label, r.label) and torch.equal(s.conf, r.conf) and torch.equal(s.unc, r.unc)
        assert torch.equal(s.class_hist, r.class_hist) and torch.equal(s.conf_hist, r.conf_hist)
        assert int(s.marginal) == int(r.marginal)
    # every source votes for a class in [0, K): a count of 1 always reaches threshold 0 and 1
    assert torch.equal(labels_at[0], labels_at[1])


# ---- 2. wide sources -------------------------------------------------------------------------------------------------------
WIDE = (256, 1, 130)                 # 52 + 1 + 26 = 79 chunks: 3 mod 4, 1 mod 3; the 1-class source is 4/5 padding


def _wide_inputs(n, K, seed, main_hw, aux_hw):
    gen = torch.Generator().manual_seed(seed)
    mains = [3 * torch.randn(n, c, *main_hw, generator=gen) + 3 * torch.randn(n, c, 1, 1, generator=gen) for c in WIDE]
    auxs = [m + 1.5 * torch.randn(m.shape, generator=gen) if aux_hw == main_hw else 3 * torch.randn(n, c, *aux_hw, generator=gen)
            for m, c in zip(mains, WIDE)]
    luts = _tables(WIDE, K, _ignore(K), gen)
    return mains, auxs, luts


@pytest.mark.parametrize("K", [5, 8])
def test_k1_wide_sources(ops, dev, sms, launches, K):
    """Sources of 256, 1 and 130 classes on 4 x 128x480 (256 tiles: 108 of the 148 CTAs run two) through the TMA kernel,
    'half' and 'prob'."""
    n, h, w = 4, 128, 480
    ignore, KT, nst = _ignore(K), (5 if K == 5 else 8), (4 if K == 5 else 3)
    n_tiles = n * -(-(h * w) // TILE)
    assert n_tiles > sms
    _ring_carry(WIDE, nst)
    mains, auxs, luts = _wide_inputs(n, K, 40 + K, (h, w), (h, w))
    with _oracle_settings(ignore):
        per = _per_source_oracle(mains, auxs, luts, K, ignore)
    md, ad = [m.to(dev) for m in mains], [a.to(dev) for a in auxs]
    for policy in ("half", "prob"):
        with _oracle_settings(ignore):
            ref = _combine(per, policy, K, ignore)
        r, ks = launches(lambda: ops.fuse_sources(md, ad, luts, policy=policy, num_classes=K, ignore_label=ignore, want_kld=True))
        _repeats(_the(ks, "fuse_sources_tma_kernel<15,2,5,%d,%d,true>" % (nst, KT)), n_tiles)
        _check_fusion(ops, r, ref, K, ignore)
        for got, want in zip(r.kld, ref["kld"]):
            torch.testing.assert_close(got.cpu(), want, rtol=RTOL, atol=3 * KLD_ATOL)


def _lowres_rows(H, W, hin):
    """lowres_plan's (fuse_launch.cuh) source rows a 960-pixel tile touches, in its fp32 arithmetic."""
    spanned = min(H, (TILE - 1) // W + 2)
    scale = np.float32(hin - 1) / np.float32(H - 1) if H > 1 else np.float32(0)
    return min(hin, int(np.float32(spanned - 1) * scale) + 3)


def _lowres_fragment(K, gk, H, W, geoms):
    """The K1-lowres instantiation mspl_fuse_sources_lowres picks: K <= 5 with every source's staged rows (plus the taps'
    one-float overread) inside 768 main / 384 aux floats runs the fixed-stride kernel, everything else the run-time one."""
    main = max(_lowres_rows(H, W, hm) * wm for (hm, wm), _ in geoms)
    aux = max(_lowres_rows(H, W, ha) * wa for _, (ha, wa) in geoms)
    fixed = K <= 5 and main + 1 <= 768 and aux + 1 <= 384
    return "fuse_sources_lowres_kernel<15,2,5,4,%d,%s,%s>" % (5 if K <= 5 else 8, str(gk).lower(), "768,384" if fixed else "0,0")


def _lowres_oracle(mains, auxs, luts, out_size, K, ignore):
    """Per-source oracle on each source's heads upsampled as the network does (O.fuse_sources_lowres, one source at a time)."""
    ups = [O.upsample_heads(m, a, out_size) for m, a in zip(mains, auxs)]
    return _per_source_oracle([u[0] for u in ups], [u[1] for u in ups], luts, K, ignore)


@pytest.mark.parametrize("K", [5, 8])
def test_k1_lowres_wide_sources(ops, dev, sms, launches, K):
    """The 256 / 1 / 130-class set through K1-lowres with ESPDNetUE heads (x2 main, x4 aux), 3 x 128x480: a stage holds 5
    classes whatever C is, so it is served.  4 x 128x480 (256 tiles); parity definition of test_fuse_sources_lowres."""
    n, (h, w) = 4, (128, 480)
    ignore = _ignore(K)
    geoms = [((h // 2, w // 2), (h // 4, w // 4))] * 3
    n_tiles = n * -(-(h * w) // TILE)
    assert n_tiles > sms
    _ring_carry(WIDE, 4)
    mains, auxs, luts = _wide_inputs(n, K, 50 + K, geoms[0][0], geoms[0][1])
    with _oracle_settings(ignore, margin=1e-5):
        per = _lowres_oracle(mains, auxs, luts, (h, w), K, ignore)
    md, ad = [m.to(dev) for m in mains], [a.to(dev) for a in auxs]
    for policy in ("half", "prob"):
        with _oracle_settings(ignore, margin=1e-5):
            ref = _combine(per, policy, K, ignore)
        r, ks = launches(lambda: ops.fuse_sources_lowres(md, ad, luts, (h, w), policy=policy, num_classes=K, ignore_label=ignore))
        _repeats(_the(ks, _lowres_fragment(K, True, h, w, geoms)), n_tiles)
        _check_fusion(ops, r, ref, K, ignore, **LOWRES_TOL)


# ---- 3. K1-lowres with a different head geometry per source ---------------------------------------------------------------
GEOM_CLASSES = (13, 20, 5, 7)                                    # 10 chunks per tile: 2 mod 4
GEOMS_480 = (((128, 240), (64, 120)),                            # ESPDNetUE
             ((64, 120), (64, 120)),
             ((32, 60), (32, 60)),
             ((86, 160), (43, 80)))                              # non-integer scales
GEOMS_512 = (((128, 256), (64, 128)),                            # x2 main: 3 rows x 256 floats > the 768-float stride
             ((64, 128), (64, 128)),
             ((32, 64), (32, 64)),
             ((86, 172), (43, 84)))


@pytest.mark.parametrize("K,width,order", [
    (5, 480, "largest_first"), (5, 480, "smallest_first"),      # fixed 768 / 384 strides
    (8, 480, "largest_first"), (8, 480, "smallest_first"),      # run-time strides
    (5, 512, "largest_first"), (5, 512, "smallest_first"),      # run-time strides (main rows too wide)
])
def test_k1_lowres_head_geometry_per_source(ops, dev, sms, launches, K, width, order):
    """Four sources with four head geometries (same_geometry = 0: each source rebuilds its taps, the stage strides are the
    maximum over sources), 8 x 256xW outputs, source 0 the largest or the smallest geometry.  The last source (86x160 /
    43x80 at W = 480: non-integer scales, different from source 0) has +60 added to its main head at a third of its
    low-resolution pixels, which puts those pixels on LowresSlowPath with that source's own geometry.  Against upsample-then-
    fuse on the CPU ('half', 'prob'; K = 8 largest-first also with ds_rate = 3), and against ops.fuse_sources on the
    GPU-upsampled heads (same labels except at counted near-ties)."""
    n, h, w = 8, 256, width
    ignore = _ignore(K)
    perm = (0, 1, 2, 3) if order == "largest_first" else (2, 1, 0, 3)
    geoms = [(GEOMS_480 if width == 480 else GEOMS_512)[i] for i in perm]
    classes = [GEOM_CLASSES[i] for i in perm]
    assert geoms[0] == max(geoms) if order == "largest_first" else geoms[0] == min(geoms)
    n_tiles = n * -(-(h * w) // TILE)
    assert n_tiles >= 6 * sms
    _ring_carry(classes, 4)
    gen = torch.Generator().manual_seed(K * 1000 + width + len(order))
    mains, auxs = [], []
    for c, ((hm, wm), (ha, wa)) in zip(classes, geoms):
        mains.append((3 * torch.randn(n, c, hm, wm, generator=gen) + 3 * torch.randn(n, c, 1, 1, generator=gen)).contiguous())
        auxs.append(3 * torch.randn(n, c, ha, wa, generator=gen))
    mains[3] += 60.0 * (torch.rand(n, 1, *geoms[3][0], generator=gen) < 1 / 3)     # a third of the last source's pixels: z > 48
    luts = _tables(classes, K, ignore, gen)
    with _oracle_settings(ignore, margin=1e-5):
        per = _lowres_oracle(mains, auxs, luts, (h, w), K, ignore)
    md, ad = [m.to(dev) for m in mains], [a.to(dev) for a in auxs]
    ups = [O.upsample_heads(m, a, (h, w)) for m, a in zip(md, ad)]
    um, ua = [u[0].contiguous() for u in ups], [u[1].contiguous() for u in ups]
    del ups
    for policy in ("half", "prob"):
        with _oracle_settings(ignore, margin=1e-5):
            ref = _combine(per, policy, K, ignore)
        ds = 3 if (K, width, order, policy) == (8, 480, "largest_first", "half") else 1
        kw = dict(policy=policy, num_classes=K, ignore_label=ignore, ds_rate=ds)
        r, ks = launches(lambda: ops.fuse_sources_lowres(md, ad, luts, (h, w), **kw))
        _repeats(_the(ks, _lowres_fragment(K, True, h, w, geoms)), n_tiles)
        _check_fusion(ops, r, ref, K, ignore, ds_rate=ds, **LOWRES_TOL)
        r2 = ops.fuse_sources(um, ua, luts, **kw)
        assert not bool(((r.label != r2.label).cpu() & ~ref["marginal"]).any())
    if (K, width) == (5, 480):
        assert _lowres_fragment(K, True, h, w, geoms).endswith("768,384>")
    else:
        assert _lowres_fragment(K, True, h, w, geoms).endswith("0,0>")


# ---- 4. the hard-label vote kernel against merge_outputs ------------------------------------------------------------------
VOTE_SHAPE = (3, 211, 997)           # 631,501 pixels: not a multiple of 4, more than one pass of 148 x 16 CTAs x 256 threads


def _vote_labels(S, K, seed):
    """(S, *VOTE_SHAPE) uint8 labels: a per-pixel favourite class most sources vote for, the rest anything in 0..255 (values
    K..255 match no class), 255 itself in every source somewhere."""
    gen = torch.Generator().manual_seed(seed)
    npix = int(np.prod(VOTE_SHAPE))
    fav = torch.randint(0, K, (npix,), generator=gen)
    p_fav = torch.rand(npix, generator=gen)                                       # per-pixel agreement
    lab = torch.where(torch.rand(S, npix, generator=gen) < p_fav,
                      fav.expand(S, npix),
                      torch.where(torch.rand(S, npix, generator=gen) < 0.5, torch.randint(0, K, (S, npix), generator=gen),
                                  torch.randint(K, 256, (S, npix), generator=gen)))
    lab[:, :: 97] = 255
    return lab.to(torch.uint8).reshape(S, *VOTE_SHAPE)


@pytest.mark.parametrize("K", [2, 5, 8])
@pytest.mark.parametrize("S", [1, 2, 4, 8, 15])
def test_vote_labels_against_merge_outputs(ops, dev, launches, S, K):
    """ops.vote_labels (ignore id K - 1, patched into the oracle) and uest_seg_multi_os.merge_outputs (the reference's
    hard-coded 4) against O.merge_outputs for every threshold form: None, 'half', 'all', '3', 'nonsense', 0..S+1, True, False."""
    from mspl_b200 import uest_seg_multi_os as U
    lab = _vote_labels(S, K, 10 * S + K)
    ld = lab.to(dev)
    ignore = K - 1
    _, ks = launches(lambda: ops.vote_labels(ld, K, None, ignore))
    _repeats(_the(ks, "vote_labels_kernel"), int(np.prod(VOTE_SHAPE)), 256)
    stack = lab.numpy()
    for thresh in [None, "half", "all", "3", "nonsense", True, False] + list(range(S + 2)):
        with _oracle_settings(255):         # no class wins with id 255: the oracle's ignored pixels, for either ignore id
            want = O.merge_outputs(stack, K, thresh)
        got = ops.vote_labels(ld, K, thresh, ignore)
        assert got.dtype == torch.uint8 and np.array_equal(got.cpu().numpy(), np.where(want == 255, ignore, want)), thresh
        got_u = U.merge_outputs(ld, K, thresh)
        assert got_u.dtype == torch.int64 and np.array_equal(got_u.cpu().numpy(), np.where(want == 255, 4, want)), thresh


def test_vote_labels_count_ceiling(ops, dev):
    """15 sources agreeing give a count of 15, the largest a 4-bit counter holds ('all' keeps the class); 16 are rejected."""
    from mspl_b200 import _lib
    n = 1001
    lab = torch.full((15, n), 3, dtype=torch.uint8)
    lab[:, 1::2] = 7
    lab[0, 2::4] = 255                                          # 14 votes: below 'all'
    got = ops.vote_labels(lab.to(dev), 8, "all", 6).cpu()
    with _oracle_settings(6):
        want = O.merge_outputs(lab.numpy(), 8, "all")
    assert np.array_equal(got.numpy(), want)
    assert int((got == 3).sum()) == len(range(0, n, 2)) - len(range(2, n, 4)) and int((got == 7).sum()) == len(range(1, n, 2))
    sixteen = torch.zeros((16, n), dtype=torch.uint8, device=dev)
    out = torch.empty(n, dtype=torch.uint8, device=dev)
    assert _lib.load().mspl_vote_labels(sixteen.data_ptr(), 16, n, 8, 16, 6, out.data_ptr(), None) == -1
    with pytest.raises(_lib.MsplError):
        ops.vote_labels(sixteen, 8, "all", 6)
