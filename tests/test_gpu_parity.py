"""-m gpu: CUDA kernels (through the C ABI) against the CPU oracle and the golden fixtures from the live reference.

Tolerances (BASELINE.json north_star): label maps / masks / histograms bit-exact except at pixels the oracle flags
as near-ties (top-2 probability margin < 1e-6), which are counted; confidences, uncertainties, thresholds and losses
within 1e-5 relative.  KLD-type quantities are differences of O(1) log terms, so they additionally get an absolute
floor of 2e-6 (the fp32 cancellation floor of the reference's own p1*logp1 - p1*logp2 sum)."""
import numpy as np
import pytest
import torch

from oracle import mspl_oracle as O

pytestmark = pytest.mark.gpu

SOURCES = (("camvid", 13), ("cityscapes", 20), ("forest", 5))
RTOL = 1e-5
KLD_ATOL = 2e-6


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ops():
    from mspl_b200 import ops as _ops
    return _ops


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x))


def _golden_sources(g, prefix=""):
    mains = [_t(g["%smain_%s" % (prefix, n)]) for n, _ in SOURCES]
    auxs = [_t(g["%saux_%s" % (prefix, n)]) for n, _ in SOURCES]
    return mains, auxs, [O.LUTS[n] for n, _ in SOURCES]


def _fuse(ops, dev, mains, auxs, luts, policy, **kw):
    return ops.fuse_sources([m.to(dev) for m in mains], [a.to(dev) for a in auxs], luts, policy=policy, **kw)


def _check_against_oracle(r, ref, policy):
    lab = r.label.cpu()
    diff = lab != ref["label"]
    n_diff, n_marg = int(diff.sum()), int(ref["marginal"].sum())
    assert not bool((diff & ~ref["marginal"]).any()), "%d label mismatches outside the %d near-tie pixels" % (n_diff, n_marg)
    ok = ~diff
    torch.testing.assert_close(r.conf.cpu()[ok], ref["conf"][ok], rtol=RTOL, atol=1e-7)
    torch.testing.assert_close(r.unc.cpu(), ref["unc"], rtol=RTOL, atol=KLD_ATOL)
    if r.kld is not None:
        for got, want in zip(r.kld, ref["kld"]):
            torch.testing.assert_close(got.cpu(), want, rtol=RTOL, atol=KLD_ATOL)
    if n_diff == 0:
        assert torch.equal(r.class_hist.cpu(), ref["class_hist"])
    assert abs(int(r.marginal.item()) - n_marg) <= max(2, n_marg // 10)
    return n_diff


@pytest.mark.parametrize("policy", ["half", "all", 1, 2, 3, "prob"])
def test_fuse_golden_3src(ops, dev, golden, policy):
    g = golden("multi_source_3src.npz")
    mains, auxs, luts = _golden_sources(g)
    r = _fuse(ops, dev, mains, auxs, luts, policy, want_kld=True)
    ref = O.fuse_sources(mains, auxs, luts, policy)
    n_diff = _check_against_oracle(r, ref, policy)
    if policy != "prob":     # labels straight from the LIVE reference (merge_outputs on its own argmax/LUT)
        want = _t(g["label_%s" % policy])
        assert int((r.label.cpu() != want).sum()) == n_diff
        if n_diff == 0:
            assert np.array_equal(r.class_hist.cpu().numpy().astype(np.float64), g["class_array_%s" % policy])
    for s, (n, _) in enumerate(SOURCES):
        torch.testing.assert_close(r.kld[s].cpu(), _t(g["kld_" + n]), rtol=RTOL, atol=KLD_ATOL)


def test_fuse_subsets_s1_s2(ops, dev, golden):
    g = golden("multi_source_3src.npz")
    mains, auxs, luts = _golden_sources(g)
    r = _fuse(ops, dev, mains[:1], auxs[:1], luts[:1], None)
    assert torch.equal(r.label.cpu(), _t(g["label_s1"]))
    r = _fuse(ops, dev, mains[:2], auxs[:2], luts[:2], "half")
    assert torch.equal(r.label.cpu(), _t(g["label_s2_half"]))
    assert np.array_equal(r.class_hist.cpu().numpy().astype(np.float64), g["class_array_s2_half"])


@pytest.mark.parametrize("tag", ["ties", "big", "onehot"])
def test_fuse_adversarial(ops, dev, golden, tag):
    """All-equal logits (pure tie-break), +-80 logits (overflow guard), one-hot +-30 (conf -> 1)."""
    g = golden("adversarial.npz")
    mains, auxs, luts = _golden_sources(g, tag + "_")
    for policy in ("half", "all"):
        r = _fuse(ops, dev, mains, auxs, luts, policy, want_kld=True)
        want = _t(g["%s_label_%s" % (tag, policy)])
        ref = O.fuse_sources(mains, auxs, luts, policy)
        if tag == "ties":
            # exact ties in z: the reference's argmax-of-softmax and our argmax-of-z both take the lowest class index
            assert torch.equal(r.label.cpu(), want)
        else:
            assert not bool(((r.label.cpu() != want) & ~ref["marginal"]).any())
        assert torch.isfinite(r.conf).all() and torch.isfinite(r.unc).all()
        for s, (n, _) in enumerate(SOURCES):
            torch.testing.assert_close(r.kld[s].cpu(), _t(g["%s_kld_%s" % (tag, n)]), rtol=RTOL, atol=2e-5 if tag == "big" else KLD_ATOL)


def test_softmax_kld_and_get_output(ops, dev, golden):
    from mspl_b200 import uest_seg_multi_os as U
    g = golden("multi_source_3src.npz")
    for n, _ in SOURCES:
        m, a = _t(g["main_" + n]), _t(g["aux_" + n])
        prob, kld = ops.softmax_kld(m.to(dev), a.to(dev))
        torch.testing.assert_close(prob.cpu(), _t(g["softmax_" + n]), rtol=RTOL, atol=1e-9)
        torch.testing.assert_close(kld.cpu(), _t(g["kld_" + n]), rtol=RTOL, atol=KLD_ATOL)
        out, k = U.get_output(lambda x: (m[1:2].to(dev), a[1:2].to(dev)), torch.zeros(1, 3, 4, 4), device=dev)
        assert out.dtype == np.float32 and out.shape == g["softmax_" + n][1].shape and k.shape == g["kld_" + n][1].shape
        np.testing.assert_allclose(out, g["softmax_" + n][1], rtol=RTOL, atol=1e-9)
    od = {"out": m[:1].to(dev), "aux": a[:1].to(dev)}
    out2, _ = U.get_output(lambda x: od, torch.zeros(1, 3, 4, 4), model_name="deeplabv3", device=dev)
    np.testing.assert_allclose(out2, g["softmax_forest"][0], rtol=RTOL, atol=1e-9)


def test_config1_crop(ops, dev, golden):
    """BASELINE config 1 fixture: random-init 20-class ESPDNetUE logits (near-uniform softmax: many near-ties)."""
    g = golden("config1_espdnetue_crop.npz")
    m, a = _t(g["main"]), _t(g["aux"])
    r = _fuse(ops, dev, [m], [a], [O.ID_CITYSCAPES_TO_GREENHOUSE], None, want_kld=True)
    ref = O.fuse_sources([m], [a], [O.ID_CITYSCAPES_TO_GREENHOUSE], None)
    want = _t(g["label"])
    diff = r.label.cpu() != want
    assert not bool((diff & ~ref["marginal"]).any())
    torch.testing.assert_close(r.kld[0].cpu(), _t(g["kld"]), rtol=RTOL, atol=KLD_ATOL)
    prob, _ = ops.softmax_kld(m.to(dev), a.to(dev))
    torch.testing.assert_close(prob.cpu(), _t(g["softmax"]), rtol=RTOL, atol=0)


def test_merge_outputs_and_helpers(dev, golden):
    from mspl_b200 import uest_seg_multi_os as U
    g = golden("multi_source_3src.npz")
    per = []
    for n, _ in SOURCES:
        amax = np.argmax(g["softmax_" + n][0], axis=0).astype(np.uint8)
        lab = U.transfer_id_to_greenhouse(O.LUTS[n], amax)
        assert np.array_equal(lab, O.LUTS[n][amax])
        per.append(lab)
        got = U.transfer_output_to_greenhouse(O.LUTS[n], g["softmax_" + n][0])
        assert got.dtype == np.float64 and np.array_equal(got, g["gh_prob_" + n][0])
    stack = np.array(per)
    for pol in (None, "half", "all", 1, 2, 3, "3", 7):
        got = U.merge_outputs(stack, 5, pol)
        assert got.dtype == np.int64 and np.array_equal(got, O.merge_outputs(stack, 5, pol))
    for pol in ("half", "all", 1, 2, 3):
        assert np.array_equal(U.merge_outputs(stack, 5, pol), g["label_%s" % pol][0])
    t = U.merge_outputs(torch.from_numpy(stack).to(dev), 5, "all")
    assert t.is_cuda and t.dtype == torch.int64


@pytest.mark.parametrize("shape", [(1, 7, 9), (2, 5, 6), (3, 16, 20)])
def test_ragged_shapes_scalar_path(ops, dev, shape):
    """H*W not a multiple of 4 -> scalar (P=1) kernels; tiny and odd sizes."""
    n, h, w = shape
    mains, auxs = [], []
    for i, (nm, c) in enumerate(SOURCES):
        m, a = O.synthetic_logits(n, c, h, w, seed=20 + i)
        mains.append(m), auxs.append(a)
    luts = [O.LUTS[nm] for nm, _ in SOURCES]
    for policy in ("half", "all", "prob"):
        r = _fuse(ops, dev, mains, auxs, luts, policy, want_kld=True)
        _check_against_oracle(r, O.fuse_sources(mains, auxs, luts, policy), policy)


def test_misaligned_views_fall_back_to_scalar(ops, dev):
    n, h, w = 2, 8, 12
    m, a = O.synthetic_logits(n, 5, h, w, seed=4)
    buf_m = torch.zeros(m.numel() + 1, device=dev)
    buf_a = torch.zeros(a.numel() + 1, device=dev)
    buf_m[1:] = m.reshape(-1).to(dev)
    buf_a[1:] = a.reshape(-1).to(dev)
    mv, av = buf_m[1:].view(n, 5, h, w), buf_a[1:].view(n, 5, h, w)       # 4-byte aligned only
    r = ops.fuse_sources([mv], [av], [O.ID_FOREST_TO_GREENHOUSE], policy=None)
    ref = O.fuse_sources([m], [a], [O.ID_FOREST_TO_GREENHOUSE], None)
    assert not bool(((r.label.cpu() != ref["label"]) & ~ref["marginal"]).any())


def test_extreme_head_disagreement_slow_path(ops, dev):
    """main and aux heads disagree by ~200 logit units: the shared-exponential form of softmax(z) underflows and the
    kernel must take its per-pixel recompute path; results still match the oracle."""
    n, h, w = 2, 16, 40
    gen = torch.Generator().manual_seed(12)
    mains, auxs = [], []
    for nm, c in SOURCES:
        im = torch.randint(0, c, (n, 1, h, w), generator=gen)
        ia = torch.randint(0, c, (n, 1, h, w), generator=gen)
        m = torch.full((n, c, h, w), -100.0).scatter_(1, im, 100.0) + torch.randn(n, c, h, w, generator=gen)
        a = torch.full((n, c, h, w), -100.0).scatter_(1, ia, 100.0) + torch.randn(n, c, h, w, generator=gen)
        mains.append(m.contiguous()), auxs.append(a.contiguous())
    luts = [O.LUTS[nm] for nm, _ in SOURCES]
    for policy in ("half", "all", "prob"):
        r = _fuse(ops, dev, mains, auxs, luts, policy, want_kld=True)
        assert torch.isfinite(r.conf).all() and torch.isfinite(r.unc).all()
        ref = O.fuse_sources(mains, auxs, luts, policy)
        lab = r.label.cpu()
        diff = lab != ref["label"]
        assert not bool((diff & ~ref["marginal"]).any())
        torch.testing.assert_close(r.conf.cpu()[~diff], ref["conf"][~diff], rtol=RTOL, atol=1e-7)
        for got, want in zip(r.kld, ref["kld"]):
            torch.testing.assert_close(got.cpu(), want, rtol=RTOL, atol=KLD_ATOL)


def test_empty_batch(ops, dev):
    m = torch.zeros(0, 5, 8, 8, device=dev)
    r = ops.fuse_sources([m], [m.clone()], [O.ID_FOREST_TO_GREENHOUSE])
    assert r.label.shape == (0, 8, 8) and int(r.class_hist.sum()) == 0


def test_rejects_cpu_tensors_and_bad_tables(ops, dev):
    m = torch.zeros(1, 5, 8, 8)
    with pytest.raises(ValueError):
        ops.fuse_sources([m], [m], [O.ID_FOREST_TO_GREENHOUSE])
    with pytest.raises(ValueError):
        ops.fuse_sources([m.to(dev)], [m.to(dev)], [[0, 1, 2, 3, 9]])
    with pytest.raises(ValueError):
        ops.fuse_sources([m.to(dev)], [m.to(dev)], [[0, 1, 2]])


@pytest.mark.parametrize("portion,ds_rate", [(0.2, 1), (0.5, 1), (0.05, 4), (1.0, 1), (0.0, 1), (1e-4, 3)])
def test_cb_thresholds_exact(ops, dev, portion, ds_rate):
    """Radix select == sort-based order statistic, bit for bit, on the very same conf values."""
    n, h, w = 3, 40, 52
    mains, auxs = [], []
    for i, (nm, c) in enumerate(SOURCES):
        m, a = O.synthetic_logits(n, c, h, w, seed=40 + i)
        mains.append(m), auxs.append(a)
    luts = [O.LUTS[nm] for nm, _ in SOURCES]
    for policy in ("half", "prob"):
        r = _fuse(ops, dev, mains, auxs, luts, policy, ds_rate=ds_rate)
        th_ref, kept_ref = O.cb_thresholds(r.label.cpu(), r.conf.cpu(), portion, ds_rate)
        th_a, kept_a = ops.cb_thresholds(r.label, r.conf, portion, ds_rate)                  # pass 0 computed standalone
        th_b, kept_b = ops.cb_thresholds(r.label, r.conf, portion, ds_rate, conf_hist=r.conf_hist)   # pass 0 fused in K1
        assert torch.equal(th_a.cpu(), th_ref) and torch.equal(kept_a.cpu(), kept_ref)
        assert torch.equal(th_b.cpu(), th_ref) and torch.equal(kept_b.cpu(), kept_ref)
        final, mask, fh = ops.apply_thresholds(r.label, r.conf, th_a)
        f_ref, m_ref = O.apply_thresholds(r.label.cpu(), r.conf.cpu(), th_ref)
        assert torch.equal(final.cpu(), f_ref) and torch.equal(mask.cpu(), m_ref)
        assert torch.equal(fh.cpu(), torch.bincount(f_ref.reshape(-1).long(), minlength=5))


def test_cb_thresholds_duplicates_and_extremes(ops, dev):
    """Heavy duplicates, zeros, ones, denormals and negative values order exactly like torch.sort."""
    gen = torch.Generator().manual_seed(9)
    label = torch.randint(0, 5, (2, 31, 33), generator=gen).to(torch.uint8)
    pool = torch.tensor([0.0, 1.0, 0.5, 0.5, 0.25, 1e-40, 3e-39, -0.25, 0.99999994, 0.33333334])
    conf = pool[torch.randint(0, pool.numel(), (2, 31, 33), generator=gen)]
    for p in (0.1, 0.37, 0.9):
        th, kept = ops.cb_thresholds(label.to(dev), conf.to(dev), p)
        th_ref, kept_ref = O.cb_thresholds(label, conf, p)
        assert torch.equal(th.cpu(), th_ref) and torch.equal(kept.cpu(), kept_ref)


@pytest.mark.parametrize("policy,portion,ds_rate", [("all", 0.2, 1), ("half", 0.2, 1), ("prob", 0.5, 1), ("half", 0.05, 4),
                                                    ("half", 1.0, 1), ("all", 0.0, 1), ("prob", 1e-4, 3), (2, 0.37, 2)])
def test_select_and_apply_matches_oracle(ops, dev, policy, portion, ds_rate):
    """Bracketed protocol (one pass + candidate list) == sort-based definition, bit for bit: thresholds of every non-ignore
    class, the final map, the mask, both histograms; and == the generic 3-pass radix protocol."""
    n, h, w = 3, 40, 52
    mains, auxs = [], []
    for i, (nm, c) in enumerate(SOURCES):
        m, a = O.synthetic_logits(n, c, h, w, seed=140 + i)
        mains.append(m), auxs.append(a)
    luts = [O.LUTS[nm] for nm, _ in SOURCES]
    r = _fuse(ops, dev, mains, auxs, luts, policy, ds_rate=ds_rate)
    lab, conf = r.label.cpu(), r.conf.cpu()
    th_ref, kept_ref = O.cb_thresholds(lab, conf, portion, ds_rate, ignore=4)
    f_ref, m_ref = O.apply_thresholds(lab, conf, th_ref)
    for hist in (None, r.conf_hist):                      # linear histogram computed stand-alone / fused into K1
        th, kept, final, mask, fh = ops.select_and_apply(r.label, r.conf, portion, ds_rate, 5, 4, conf_hist=hist, want_mask=True)
        assert torch.equal(th.cpu(), th_ref) and torch.equal(kept.cpu(), kept_ref)
        assert torch.equal(final.cpu(), f_ref) and torch.equal(mask.cpu(), m_ref)
        assert torch.equal(fh.cpu(), torch.bincount(f_ref.reshape(-1).long(), minlength=5))
    assert int(r.conf_hist.abs().sum()) == 0              # consumed
    # a (trivial) all-reduce hook switches the final counts to this rank's saved copy of the histogram: same results
    th, kept, final, mask, fh = ops.select_and_apply(r.label, r.conf, portion, ds_rate, 5, 4, all_reduce=lambda t: t, want_mask=True)
    assert torch.equal(th.cpu(), th_ref) and torch.equal(final.cpu(), f_ref) and torch.equal(mask.cpu(), m_ref)
    assert torch.equal(fh.cpu(), torch.bincount(f_ref.reshape(-1).long(), minlength=5))
    th_radix, kept_radix = ops.cb_thresholds_radix(r.label, r.conf, portion, ds_rate)
    th_all, kept_all = ops.cb_thresholds(r.label, r.conf, portion, ds_rate)                # every class resolved
    assert torch.equal(th_radix, th_all) and torch.equal(kept_radix, kept_all)
    assert torch.equal(th_all.cpu(), O.cb_thresholds(lab, conf, portion, ds_rate)[0])
    assert torch.equal(th_all[:4].cpu(), th_ref[:4])


def test_select_and_apply_degenerate_and_large(ops, dev):
    """Every pixel a candidate (one shared conf value), values outside [0,1], NaN-free extremes, and a map large enough for
    several grid-stride iterations and many staging flushes per warp."""
    gen = torch.Generator().manual_seed(19)
    cases = []
    label = torch.randint(0, 5, (2, 64, 80), generator=gen).to(torch.uint8)
    cases.append((label, torch.full((2, 64, 80), 0.7312), 0.3))                              # one value: all candidates
    pool = torch.tensor([0.0, 1.0, 0.5, 0.5, 0.25, 1e-40, 3e-39, -0.25, 0.99999994, 0.33333334, 2.5, 1e30, -1e30, 4.8828125e-4])
    cases.append((label, pool[torch.randint(0, pool.numel(), (2, 64, 80), generator=gen)], 0.37))
    big_label = torch.randint(0, 5, (12, 512, 1024), generator=gen).to(torch.uint8)           # 6.3 Mpix > one grid sweep
    big_conf = torch.rand((12, 512, 1024), generator=gen)
    big_conf[:, ::2] = (big_conf[:, ::2] * 64).floor() / 64                                  # heavy duplicates on bin edges
    cases.append((big_label, big_conf, 0.2))
    cases.append((big_label, torch.full((12, 512, 1024), 0.4), 0.5))                         # 6.3 M candidates
    for label, conf, p in cases:
        th_ref, kept_ref = O.cb_thresholds(label, conf, p, ignore=4)
        f_ref, m_ref = O.apply_thresholds(label, conf, th_ref)
        th, kept, final, mask, fh = ops.select_and_apply(label.to(dev), conf.to(dev), p, 1, 5, 4, want_mask=True)
        assert torch.equal(th.cpu(), th_ref) and torch.equal(kept.cpu(), kept_ref)
        assert torch.equal(final.cpu(), f_ref) and torch.equal(mask.cpu(), m_ref)
        assert torch.equal(fh.cpu(), torch.bincount(f_ref.reshape(-1).long(), minlength=5))
        th_all, _ = ops.cb_thresholds(label.to(dev), conf.to(dev), p)
        assert torch.equal(th_all.cpu(), O.cb_thresholds(label, conf, p)[0])


def test_select_and_apply_odd_sizes(ops, dev):
    """Pixel counts that are not multiples of 4 and unaligned views take the scalar path."""
    gen = torch.Generator().manual_seed(23)
    for shape in ((1, 7, 9), (3, 5, 7), (2, 33, 31)):
        label = torch.randint(0, 5, shape, generator=gen).to(torch.uint8)
        conf = torch.rand(shape, generator=gen)
        th_ref, kept_ref = O.cb_thresholds(label, conf, 0.3, ignore=4)
        f_ref, m_ref = O.apply_thresholds(label, conf, th_ref)
        th, kept, final, mask, fh = ops.select_and_apply(label.to(dev), conf.to(dev), 0.3, 1, 5, 4, want_mask=True)
        assert torch.equal(th.cpu(), th_ref) and torch.equal(kept.cpu(), kept_ref)
        assert torch.equal(final.cpu(), f_ref) and torch.equal(mask.cpu(), m_ref)


def test_bracketed_protocol_sharded_raw_abi(ops, dev):
    """Emulates 2 ranks on one GPU through the raw C ABI: every rank keeps its own state / candidate list / final histogram,
    the linear histogram and each candidate pass's histogram are summed over the ranks (the all-reduce) before each rank's
    select, and the final class counts are read off each rank's local histogram.  Result == unsharded == oracle."""
    from mspl_b200 import _lib
    import ctypes
    lib = _lib.load()
    gen = torch.Generator().manual_seed(29)
    K, h, w = 5, 48, 64
    label = torch.randint(0, K, (6, h, w), generator=gen).to(torch.uint8).to(dev)
    conf = torch.rand((6, h, w), generator=gen).to(dev)
    conf[0, :4] = 1.0                                          # some pixels exactly at the "threshold 1.0" of tiny classes
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None

    class Rank:
        def __init__(self, lab, cf):
            self.lab, self.cf = lab.contiguous(), cf.contiguous()
            self.state = torch.zeros(lib.mspl_radix_state_bytes(K), dtype=torch.uint8, device=dev)
            self.thresh = torch.empty(K, dtype=torch.float32, device=dev)
            self.bracket = torch.empty((K, 2), dtype=torch.float32, device=dev)
            self.kept = torch.zeros(K, dtype=torch.int64, device=dev)
            self.hist = torch.zeros((K, 2048), dtype=torch.int64, device=dev)
            self.fh = torch.zeros(K, dtype=torch.int64, device=dev)
            self.final = torch.empty_like(self.lab)
            self.cand = torch.empty(self.lab.numel(), dtype=torch.int32, device=dev)
            self.count = torch.zeros((), dtype=torch.int64, device=dev)

    def all_reduce(ranks):
        total = sum(r.hist for r in ranks)
        for r in ranks:
            r.hist.copy_(total)

    for portion in (0.25, 1e-5):                               # 1e-5: every class has j == 0 -> threshold 1.0
        ranks = [Rank(label[:2], conf[:2]), Rank(label[2:], conf[2:])]
        for r in ranks:
            _lib.check(lib.mspl_conf_hist(p(r.lab), p(r.cf), r.lab.numel(), h * w, K, p(r.hist), 1, st), "conf_hist")
            r.local = r.hist.clone()
        all_reduce(ranks)
        for r in ranks:
            _lib.check(lib.mspl_bracket_select(p(r.hist), K, portion, 4, p(r.state), p(r.bracket), p(r.thresh), p(r.kept), p(r.local),
                                               p(r.fh), st), "bracket_select")
            _lib.check(lib.mspl_bracket_classify(p(r.lab), p(r.cf), p(r.bracket), r.lab.numel(), K, 4, p(r.final), None, None,
                                                 p(r.cand), p(r.count), st), "classify")
        for ps in range(3):
            for r in ranks:
                _lib.check(lib.mspl_cand_hist_pass(p(r.lab), p(r.cf), p(r.cand), p(r.count), h * w, K, ps, p(r.state), p(r.hist), 1, st),
                           "cand_hist")
            all_reduce(ranks)
            for r in ranks:
                _lib.check(lib.mspl_cand_select(p(r.hist), K, ps, p(r.state), p(r.thresh), None, -1, st), "cand_select")
        for r in ranks:
            _lib.check(lib.mspl_cand_apply(p(r.lab), p(r.cf), p(r.thresh), p(r.cand), p(r.count), K, 4, p(r.final), None, p(r.fh), st),
                       "cand_apply")
        th_ref, kept_ref = O.cb_thresholds(label.cpu(), conf.cpu(), portion, ignore=4)
        f_ref, _ = O.apply_thresholds(label.cpu(), conf.cpu(), th_ref)
        for r in ranks:
            assert torch.equal(r.thresh.cpu(), th_ref) and torch.equal(r.kept.cpu(), kept_ref)
            assert torch.equal(r.fh, torch.bincount(r.final.reshape(-1).long(), minlength=K))       # per-rank counts are local
        assert torch.equal(torch.cat([r.final for r in ranks]).cpu(), f_ref)
        assert torch.equal(sum(r.fh for r in ranks).cpu(), torch.bincount(f_ref.reshape(-1).long(), minlength=K))
        if portion == 0.25:
            assert sum(int(r.count) for r in ranks) < label.numel() // 100      # candidates are a tiny fraction of the pixels
        th1, kept1, final1, _, fh1 = ops.select_and_apply(label, conf, portion, 1, K, 4)
        assert torch.equal(th1, ranks[0].thresh) and torch.equal(final1.cpu(), f_ref)
        assert torch.equal(fh1, sum(r.fh for r in ranks))


def test_thresholds_vs_oracle_conf(ops, dev):
    """End to end against the oracle's own conf: thresholds within 1e-5 relative; final labels equal except at
    near-tie pixels and pixels whose conf sits within 1e-5 relative of its class threshold."""
    n, h, w = 4, 64, 96
    mains, auxs = [], []
    for i, (nm, c) in enumerate(SOURCES):
        m, a = O.synthetic_logits(n, c, h, w, seed=60 + i)
        mains.append(m), auxs.append(a)
    luts = [O.LUTS[nm] for nm, _ in SOURCES]
    r = _fuse(ops, dev, mains, auxs, luts, "half")
    ref = O.fuse_sources(mains, auxs, luts, "half")
    th, _ = ops.cb_thresholds(r.label, r.conf, 0.2, conf_hist=r.conf_hist)
    th_ref, _ = O.cb_thresholds(ref["label"], ref["conf"], 0.2)
    torch.testing.assert_close(th.cpu(), th_ref, rtol=RTOL, atol=0)
    final, _, _ = ops.apply_thresholds(r.label, r.conf, th)
    f_ref, _ = O.apply_thresholds(ref["label"], ref["conf"], th_ref)
    near_thresh = (ref["conf"] - th_ref[ref["label"].long()]).abs() <= 2e-5 * th_ref[ref["label"].long()]
    bad = (final.cpu() != f_ref) & ~ref["marginal"] & ~near_thresh
    assert not bool(bad.any())


@pytest.mark.parametrize("tag", ["flat", "normal"])
def test_fused_loss_golden(ops, dev, golden, tag):
    g = golden("loss_k5.npz")
    main, aux, target, cw = _t(g["main"]), _t(g["aux"]), _t(g["target"]), _t(g["cw_" + tag])
    md, ad = main.to(dev).requires_grad_(True), aux.to(dev).requires_grad_(True)
    loss, parts = ops.uw_ce_loss(md, ad, target.to(dev), cw.to(dev), return_parts=True)
    loss.backward()
    want = float(g["loss_" + tag])
    assert abs(loss.item() - want) <= RTOL * abs(want)
    assert abs(parts[0].item() - (20 * parts[1].item() + parts[2].item())) <= 1e-5 * abs(want)
    scale = float(np.abs(g["grad_main_" + tag]).max())
    torch.testing.assert_close(md.grad.cpu(), _t(g["grad_main_" + tag]), rtol=1e-4, atol=1e-5 * scale)
    torch.testing.assert_close(ad.grad.cpu(), _t(g["grad_aux_" + tag]), rtol=1e-4, atol=1e-5 * scale)
    # upstream gradient != 1 goes through the on-device scale kernel
    md2, ad2 = main.to(dev).requires_grad_(True), aux.to(dev).requires_grad_(True)
    (ops.uw_ce_loss(md2, ad2, target.to(dev), cw.to(dev)) * 0.25).backward()
    torch.testing.assert_close(md2.grad, md.grad * 0.25, rtol=1e-6, atol=0)
    torch.testing.assert_close(ad2.grad, ad.grad * 0.25, rtol=1e-6, atol=0)


def test_fused_loss_fp64_oracle_and_determinism(ops, dev):
    """Gradients against the fp64 oracle (tighter than fp32-vs-fp32) and bitwise run-to-run determinism."""
    b, k, h, w = 4, 5, 36, 44
    main, aux = O.synthetic_logits(b, k, h, w, seed=77)
    target = torch.randint(0, k, (b, h, w), generator=torch.Generator().manual_seed(1))
    cw = torch.tensor([0.0, 2.5, 1.0, 4.0, 0.0])
    l64, gm64, ga64 = O.training_loss_and_grads(main, aux, target, cw, dtype=torch.float64)
    out3, dm, da = ops.uw_ce_fwd_bwd(main.to(dev), aux.to(dev), target.to(dev), cw.to(dev))
    assert abs(out3[0].item() - l64.item()) <= RTOL * abs(l64.item())
    scale = float(gm64.abs().max())
    torch.testing.assert_close(dm.cpu().double(), gm64, rtol=2e-5, atol=2e-6 * scale)
    torch.testing.assert_close(da.cpu().double(), ga64, rtol=2e-5, atol=2e-6 * scale)
    out3b, dmb, dab = ops.uw_ce_fwd_bwd(main.to(dev), aux.to(dev), target.to(dev), cw.to(dev))
    assert torch.equal(out3, out3b) and torch.equal(dm, dmb) and torch.equal(da, dab)
    out3f, none_m, none_a = ops.uw_ce_fwd_bwd(main.to(dev), aux.to(dev), target.to(dev), cw.to(dev), backward=False)
    assert none_m is None and none_a is None and torch.equal(out3f, out3)
    # data-parallel form: two half-batches with the GLOBAL pixel count sum to the full-batch loss and grads
    norm = b * h * w
    o_a, dm_a, _ = ops.uw_ce_fwd_bwd(main[:2].to(dev), aux[:2].to(dev), target[:2].to(dev), cw.to(dev), norm_pixels=norm)
    o_b, dm_b, _ = ops.uw_ce_fwd_bwd(main[2:].to(dev), aux[2:].to(dev), target[2:].to(dev), cw.to(dev), norm_pixels=norm)
    assert abs((o_a[0] + o_b[0]).item() - out3[0].item()) <= 1e-6 * abs(out3[0].item())
    torch.testing.assert_close(torch.cat([dm_a, dm_b]), dm, rtol=1e-6, atol=0)


@pytest.mark.parametrize("shape", [(4, 5, 36, 44), (2, 5, 31, 7), (3, 8, 16, 18), (1, 1, 8, 8)])
def test_fused_loss_uint8_targets(ops, dev, shape):
    """uint8 class indices (the format the label maps are generated and stored in) give the same bits as int64 targets,
    for the full-resolution and the fused-upsample kernels, aligned (vector) and unaligned (scalar) target loads alike;
    255 -- outside [0,K) for either dtype -- contributes like a zero-weight class."""
    b, k, h, w = shape
    main, aux = O.synthetic_logits(b, k, h, w, seed=91)
    target = torch.randint(0, k, (b, h, w), generator=torch.Generator().manual_seed(5))
    target[0, 0, :3] = 255
    cw = torch.rand(k, generator=torch.Generator().manual_seed(6)) + 0.5
    m, a, t64, c = main.to(dev), aux.to(dev), target.to(dev), cw.to(dev)
    t8 = t64.to(torch.uint8)
    want = ops.uw_ce_fwd_bwd(m, a, t64, c)
    got = ops.uw_ce_fwd_bwd(m, a, t8, c)
    for x, y in zip(want, got):
        assert torch.equal(x, y)
    # against the oracle: pixels labelled 255 carry weight 0, i.e. behave like a class whose weight is zero
    t_or = target.clone()
    cw_or = torch.cat([cw, torch.zeros(1)])
    t_or[target == 255] = k
    pad = torch.full((b, 1, h, w), -1e4)            # an extra class no pixel can prefer: softmax over K unchanged
    l64, gm64, _ = O.training_loss_and_grads(torch.cat([main, pad], 1), torch.cat([aux, pad], 1), t_or, cw_or, dtype=torch.float64)
    assert abs(got[0][0].item() - l64.item()) <= RTOL * abs(l64.item())
    torch.testing.assert_close(got[1].cpu().double(), gm64[:, :k], rtol=2e-5, atol=2e-6 * float(gm64.abs().max()))
    # an offset view: targets no longer 4-byte aligned -> the scalar-load instantiation
    flat = torch.zeros(t8.numel() + 1, dtype=torch.uint8, device=dev)
    flat[1:] = t8.reshape(-1)
    got_off = ops.uw_ce_fwd_bwd(m, a, flat[1:].view(b, h, w), c)
    torch.testing.assert_close(got_off[0], want[0], rtol=1e-6, atol=0)
    torch.testing.assert_close(got_off[1], want[1], rtol=1e-6, atol=1e-12)
    # autograd route and the fused-upsample kernel
    md, ad = m.clone().requires_grad_(True), a.clone().requires_grad_(True)
    ops.uw_ce_loss(md, ad, t8, c).backward()
    assert torch.equal(md.grad, want[1]) and torch.equal(ad.grad, want[2])
    if h >= 4 and w >= 4:
        ml, al = m[:, :, ::2, ::2].contiguous(), a[:, :, ::4, ::4].contiguous()
        for x, y in zip(ops.uw_ce_lowres_fwd_bwd(ml, al, t64, c), ops.uw_ce_lowres_fwd_bwd(ml, al, t8, c)):
            assert torch.equal(x, y)
    with pytest.raises(ValueError):
        ops.uw_ce_fwd_bwd(m, a, t64.to(torch.int32), c)


@pytest.mark.parametrize("shape,dtype", [((4, 5, 36, 44), torch.int64), ((4, 5, 36, 44), torch.uint8), ((2, 5, 31, 7), torch.int64),
                                         ((3, 8, 16, 18), torch.uint8), ((1, 2, 8, 8), torch.int64), ((6, 5, 256, 480), torch.uint8)])
def test_fused_loss_with_iou_counts(ops, dev, shape, dtype):
    """One launch = the loss AND the counts of the training loop's next statement, miou_class.get_iou(pred, labels)
    (uest_seg_multi_os.py:1032): counts bit-equal to the oracle's restatement of MIOU.get_iou and to the stand-alone metric
    kernel (itself pinned to the live reference), loss and gradients bit-equal to the launch without the counts."""
    b, k, h, w = shape
    main, aux = O.synthetic_logits(b, k, h, w, seed=17)
    main[0, :, 0, :2] = 1.25                                    # argmax ties -> first index
    target = torch.randint(0, k, (b, h, w), generator=torch.Generator().manual_seed(8))
    target[0, 0, 2:5] = 255                                     # wraps to 0 after the +1 shift: dropped
    if k < 8:
        target[0, 1, :3] = k                                    # a class id outside histc's range: not counted as mask
    cw = torch.rand(k, generator=torch.Generator().manual_seed(9)) + 0.5
    m, a, t, c = main.to(dev), aux.to(dev), target.to(dev).to(dtype), cw.to(dev)
    counts = torch.zeros((3, k), dtype=torch.int64, device=dev)
    got = ops.uw_ce_fwd_bwd(m, a, t, c, iou_counts=counts)
    plain = ops.uw_ce_fwd_bwd(m, a, t, c)
    for x, y in zip(got, plain):
        assert torch.equal(x, y)
    inter, union = O.miou_get_iou(main, target, num_classes=k)
    alone = ops.miou_counts(m, target.to(dev), k)
    assert torch.equal(counts, alone)
    np.testing.assert_array_equal(counts[0].cpu().numpy().astype(np.float32), inter)
    np.testing.assert_array_equal((counts[1] + counts[2] - counts[0]).cpu().numpy().astype(np.float32) + np.float32(1e-6), union)
    # accumulation (+=) and forward-only launches
    ops.uw_ce_fwd_bwd(m, a, t, c, backward=False, iou_counts=counts)
    assert torch.equal(counts, 2 * alone)
    with pytest.raises(ValueError):
        ops.uw_ce_fwd_bwd(m, a, t, c, iou_counts=torch.zeros((3, k + 1), dtype=torch.int64, device=dev))


def test_fused_loss_module_tracks_epoch_iou(dev):
    """FusedUncertaintyWeightedLoss(track_iou=True) over several batches == the reference loop's meters
    (inter_meter.sum / (union_meter.sum + 1e-10), uest_seg_multi_os.py:1032-1049) fed by the oracle's MIOU.get_iou."""
    from mspl_b200.loss_fns.segmentation_loss import FusedUncertaintyWeightedLoss
    k, h, w = 5, 40, 48
    crit = FusedUncertaintyWeightedLoss(k, torch.ones(k, device=dev), 4, device=dev, track_iou=True)
    inter_sum, union_sum = np.zeros(k, np.float32), np.zeros(k, np.float32)
    for step in range(3):
        main, aux = O.synthetic_logits(2, k, h, w, seed=30 + step)
        target = torch.randint(0, k, (2, h, w), generator=torch.Generator().manual_seed(step))
        md = main.to(dev).requires_grad_(True)
        crit(md, aux.to(dev), target.to(dev)).backward()
        assert md.grad is not None
        i, u = O.miou_get_iou(main, target, num_classes=k)
        inter_sum += i
        union_sum += u
    np.testing.assert_allclose(crit.iou(), inter_sum / (union_sum + 1e-10), rtol=1e-6)
    crit.reset_iou()
    assert crit.iou_counts is None


def test_fused_training_step_matches_live_reference_golden(dev, golden):
    """FusedUncertaintyWeightedLoss(track_iou=True) against what the LIVE reference's training-loop statements produced for
    three batches (tests/golden/train_step.npz: loss, gradients, and the epoch IoU from its two AverageMeters,
    uest_seg_multi_os.py:1020-1049).  The labels are fed as they are -- uint8, with the 255s the metric drops: a 255 weighs
    nothing in the fused loss, exactly like the ignore class the reference had to remap it to for torch.gather."""
    from mspl_b200.loss_fns.segmentation_loss import FusedUncertaintyWeightedLoss
    g = golden("train_step.npz")
    for as_u8 in (False, True):
        crit = FusedUncertaintyWeightedLoss(5, _t(g["class_weights"]).clone().to(dev), ignore_idx=4, device=dev, track_iou=True)
        for i in range(3):
            md, ad = _t(g["main_%d" % i]).to(dev).requires_grad_(True), _t(g["aux_%d" % i]).to(dev).requires_grad_(True)
            labels = _t(g["labels_%d" % i]).to(dev)
            loss = crit(md, ad, labels.to(torch.uint8) if as_u8 else labels)
            loss.backward()
            want = float(g["loss_%d" % i])
            assert abs(loss.item() - want) <= RTOL * abs(want)
            scale = float(np.abs(g["grad_main_%d" % i]).max())
            torch.testing.assert_close(md.grad.cpu(), _t(g["grad_main_%d" % i]), rtol=1e-4, atol=1e-5 * scale)
            torch.testing.assert_close(ad.grad.cpu(), _t(g["grad_aux_%d" % i]), rtol=1e-4, atol=1e-5 * scale)
        np.testing.assert_allclose(crit.iou(), g["iou"], rtol=1e-6, atol=0)
        assert abs(float(crit.iou()[[1, 2, 3]].mean() * 100) - float(g["miou"])) < 1e-3
        assert crit.iou_batches == 3 and int(crit.iou_counts[2].sum()) == 3 * 2 * 24 * 40 - 4


LOWRES_GEOMETRIES = [
    # (B, K, H, W, (hm, wm), (ha, wa))
    (2, 5, 256, 480, (128, 240), (64, 120)),        # ESPDNetUE on the benchmark crop: x2 main head, x4 aux head, 8-row tiles
    (3, 3, 37, 50, (19, 25), (10, 13)),             # odd sizes, non-integer scales, partial last tile
    (2, 5, 24, 32, (24, 32), (12, 16)),             # main head already at full resolution
    (1, 8, 20, 44, (7, 11), (3, 5)),                # K = 8, large scale factors
    (2, 2, 9, 1, (5, 1), (3, 1)),                   # single column
    (1, 5, 512, 1024, (256, 512), (128, 256)),      # stress size: only 2-row tiles fit -> an aux row gets shares from 3+ tiles
]


@pytest.mark.parametrize("geom", LOWRES_GEOMETRIES)
def test_fused_upsample_loss_matches_oracle(ops, dev, geom):
    """K4-lowres == F.interpolate(bilinear, align_corners=True) + training loss + autograd through both (the oracle's
    definition): loss 1e-5 relative, gradients w.r.t. the PRE-upsample tensors against the fp64 oracle; bitwise reproducible."""
    b, k, h, w, (hm, wm), (ha, wa) = geom
    gen = torch.Generator().manual_seed(h * 131 + w)
    main_lr = 3.0 * torch.randn(b, k, hm, wm, generator=gen)
    aux_lr = main_lr.new_empty(b, k, ha, wa).normal_(0, 3.0, generator=gen)
    target = torch.randint(0, k, (b, h, w), generator=gen)
    cw = torch.rand(k, generator=gen) * 3
    cw[k - 1] = 0.0
    l64, gm64, ga64 = O.training_loss_lowres_and_grads(main_lr, aux_lr, target, cw, dtype=torch.float64)
    l32, _, _ = O.training_loss_lowres_and_grads(main_lr, aux_lr, target, cw)
    out3, dm, da = ops.uw_ce_lowres_fwd_bwd(main_lr.to(dev), aux_lr.to(dev), target.to(dev), cw.to(dev))
    assert abs(out3[0].item() - l64.item()) <= RTOL * abs(l64.item())
    assert abs(out3[0].item() - l32.item()) <= RTOL * abs(l32.item())
    assert abs(out3[0].item() - (20 * out3[1].item() + out3[2].item())) <= 1e-5 * abs(l64.item())
    # a low-resolution gradient is a weighted sum of up to (2*scale)^2 per-pixel fp32 gradients of mixed sign: the absolute
    # floor is 5e-5 of the largest gradient instead of the 1e-5 used for the per-pixel gradients of the full-resolution K4
    scale = float(max(gm64.abs().max(), ga64.abs().max()))
    torch.testing.assert_close(dm.cpu().double(), gm64, rtol=1e-4, atol=5e-5 * scale)
    torch.testing.assert_close(da.cpu().double(), ga64, rtol=1e-4, atol=5e-5 * scale)
    out3b, dmb, dab = ops.uw_ce_lowres_fwd_bwd(main_lr.to(dev), aux_lr.to(dev), target.to(dev), cw.to(dev))
    assert torch.equal(out3, out3b)
    if w <= 480 and max((h - 1) / max(hm - 1, 1), (h - 1) / max(ha - 1, 1)) <= 4.1:
        # 8-row tiles and row scale factors up to x4 (ESPDNetUE's heads): every low-resolution element gets at most two
        # shares, and two adds onto a zeroed element commute -> bit-reproducible
        assert torch.equal(dm, dmb) and torch.equal(da, dab)
    else:
        # larger factors: a low-resolution row's footprint (2 x scale output rows) can straddle three tiles, and the order of
        # their fp32 adds is not fixed (as in ATen's upsample backward): equal to rounding, not bit for bit
        torch.testing.assert_close(dm, dmb, rtol=1e-5, atol=1e-6 * scale)
        torch.testing.assert_close(da, dab, rtol=1e-5, atol=1e-6 * scale)
    out3f, none_m, none_a = ops.uw_ce_lowres_fwd_bwd(main_lr.to(dev), aux_lr.to(dev), target.to(dev), cw.to(dev), backward=False)
    assert none_m is None and none_a is None and torch.equal(out3f, out3)
    # the same numbers as upsampling on the device and running the full-resolution K4
    mu, au = O.upsample_heads(main_lr.to(dev).requires_grad_(True), aux_lr.to(dev), (h, w))
    full, _, _ = ops.uw_ce_fwd_bwd(mu.detach().contiguous(), au.contiguous(), target.to(dev), cw.to(dev), backward=False)
    assert abs(full[0].item() - out3[0].item()) <= RTOL * abs(full[0].item())


def test_fused_upsample_loss_autograd_and_module(ops, dev):
    from mspl_b200.loss_fns.segmentation_loss import FusedUncertaintyWeightedLoss, FusedUpsampleUncertaintyWeightedLoss
    b, k, h, w = 2, 5, 64, 96
    gen = torch.Generator().manual_seed(91)
    main_lr, aux_lr = 2.0 * torch.randn(b, k, h // 2, w // 2, generator=gen), 2.0 * torch.randn(b, k, h // 4, w // 4, generator=gen)
    target = torch.randint(0, k, (b, h, w), generator=gen).to(dev)
    ml, al = main_lr.to(dev).requires_grad_(True), aux_lr.to(dev).requires_grad_(True)
    crit = FusedUpsampleUncertaintyWeightedLoss(k, class_weights=torch.ones(k, device=dev), ignore_idx=4, device=dev)
    (crit(ml, al, target) * 0.5).backward()
    # reference route on the device: F.interpolate (autograd) + the full-resolution fused loss
    ml2, al2 = main_lr.to(dev).requires_grad_(True), aux_lr.to(dev).requires_grad_(True)
    mu, au = O.upsample_heads(ml2, al2, (h, w))
    crit_full = FusedUncertaintyWeightedLoss(k, class_weights=torch.ones(k, device=dev), ignore_idx=4, device=dev)
    (crit_full(mu, au, target) * 0.5).backward()
    scale = float(ml2.grad.abs().max())
    torch.testing.assert_close(ml.grad, ml2.grad, rtol=1e-4, atol=5e-5 * scale)
    torch.testing.assert_close(al.grad, al2.grad, rtol=1e-4, atol=5e-5 * scale)
    torch.testing.assert_close(crit.last_parts, crit_full.last_parts, rtol=RTOL, atol=1e-7)
    with pytest.raises(NotImplementedError):        # a source larger than the output is not an upsample
        ops.uw_ce_loss_lowres(torch.zeros(1, 5, 80, 96, device=dev), al[:1].detach(), target[:1], torch.ones(5, device=dev))


def test_fused_upsample_loss_trains_a_network(dev):
    """The training-step wiring: forward_lowres() hands the loss the heads a network holds before its closing upsample
    (the interception ESPDNetUE needs, model/segmentation/espdnet_ue.py:301-302) and the parameter gradients equal those of
    the ordinary route (network upsamples, autograd runs upsample_bilinear2d_backward, full-resolution fused loss)."""
    import torch.nn.functional as F
    from mspl_b200.lowres import forward_lowres
    from mspl_b200.loss_fns.segmentation_loss import FusedUncertaintyWeightedLoss, FusedUpsampleUncertaintyWeightedLoss

    class TwoHeads(torch.nn.Module):                   # the closing statements of ESPDNetwithUncertaintyEstimation.forward
        def __init__(self):
            super().__init__()
            self.main = torch.nn.Conv2d(3, 5, 3, stride=2, padding=1)
            self.aux = torch.nn.Conv2d(3, 5, 5, stride=4, padding=2)

        def forward(self, x):
            size = x.shape[-2:]
            return (F.interpolate(self.main(x), size=size, mode='bilinear', align_corners=True),
                    F.interpolate(self.aux(x), size=size, mode='bilinear', align_corners=True))

    torch.manual_seed(4)
    net = TwoHeads().to(dev)
    x = torch.randn(2, 3, 48, 64, device=dev)
    labels = torch.randint(0, 5, (2, 48, 64), device=dev)
    cw = torch.ones(5, device=dev)
    pred, pred_aux = net(x)
    FusedUncertaintyWeightedLoss(5, cw.clone(), 4, dev)(pred, pred_aux, labels).backward()
    want = [p.grad.clone() for p in net.parameters()]
    net.zero_grad()
    heads = forward_lowres(net, x)
    assert heads is not None and heads[0].shape[-2:] == (24, 32) and heads[1].shape[-2:] == (12, 16)
    FusedUpsampleUncertaintyWeightedLoss(5, cw.clone(), 4, dev)(heads[0], heads[1], labels).backward()
    for p, g in zip(net.parameters(), want):
        torch.testing.assert_close(p.grad, g, rtol=1e-4, atol=1e-5 * float(g.abs().max()))


@pytest.mark.parametrize("tag", ["flat", "normal"])
def test_reference_named_modules(dev, golden, tag):
    """PixelwiseKLD / UncertaintyWeightedSegmentationLoss used exactly as uest_seg_multi_os.py:1020-1023 uses them."""
    from mspl_b200.loss_fns.segmentation_loss import (FusedUncertaintyWeightedLoss, PixelwiseKLD,
                                                      UncertaintyWeightedSegmentationLoss)
    g = golden("loss_k5.npz")
    main, aux, target = _t(g["main"]).to(dev), _t(g["aux"]).to(dev), _t(g["target"]).to(dev)
    cw_in = torch.ones(5, device=dev) if tag == "flat" else torch.tensor([0.0, 3.1, 7.7, 2.2, 9.0], device=dev)
    criterion = UncertaintyWeightedSegmentationLoss(5, class_weights=cw_in, ignore_idx=4, device=dev)
    assert criterion.class_weights is cw_in and cw_in[4].item() == 0.0          # in-place zeroing quirk kept
    pred, pred_aux = main.clone().requires_grad_(True), aux.clone().requires_grad_(True)
    kld = PixelwiseKLD()(pred, pred_aux)
    loss = criterion(pred + 0.5 * pred_aux, target, kld) * 20 + kld.mean()
    loss.backward()
    want = float(g["loss_" + tag])
    assert abs(loss.item() - want) <= RTOL * abs(want)
    scale = float(np.abs(g["grad_main_" + tag]).max())
    torch.testing.assert_close(pred.grad.cpu(), _t(g["grad_main_" + tag]), rtol=1e-4, atol=1e-5 * scale)
    torch.testing.assert_close(pred_aux.grad.cpu(), _t(g["grad_aux_" + tag]), rtol=1e-4, atol=1e-5 * scale)
    # the two modules on their own, with independent inputs
    p = main.clone().requires_grad_(True)
    u = _t(g["uw_u_" + tag]).to(dev).requires_grad_(True)
    l2 = criterion(p, target, u)
    l2.backward()
    assert abs(l2.item() - float(g["uw_loss_" + tag])) <= RTOL * abs(float(g["uw_loss_" + tag]))
    s2 = float(np.abs(g["uw_grad_pred_" + tag]).max())
    torch.testing.assert_close(p.grad.cpu(), _t(g["uw_grad_pred_" + tag]), rtol=1e-4, atol=1e-5 * s2)
    torch.testing.assert_close(u.grad.cpu(), _t(g["uw_grad_u_" + tag]), rtol=1e-4, atol=1e-5 * float(np.abs(g["uw_grad_u_" + tag]).max()))
    d1, d2 = main.clone().requires_grad_(True), aux.clone().requires_grad_(True)
    kl = PixelwiseKLD()(d1, d2)
    kl.backward(_t(g["kld_upstream"]).to(dev))
    torch.testing.assert_close(kl.detach().cpu(), _t(g["kld"]), rtol=RTOL, atol=KLD_ATOL)
    torch.testing.assert_close(d1.grad.cpu(), _t(g["kld_grad1"]), rtol=1e-4, atol=2e-6)
    torch.testing.assert_close(d2.grad.cpu(), _t(g["kld_grad2"]), rtol=1e-4, atol=2e-6)
    fused = FusedUncertaintyWeightedLoss(5, class_weights=cw_in.clone(), ignore_idx=4, device=dev)
    lf = fused(main.clone().requires_grad_(True), aux.clone(), target)
    assert abs(lf.item() - want) <= RTOL * abs(want)


def test_full_size_properties(ops, dev):
    """480x256 images at full resolution (too slow for the CPU oracle in bulk): size-independent properties --
    sharding invariance (two halves == whole, histograms add up exactly), class_hist == bincount(label),
    conf_hist row sums == kept counts, thresholded labels only ever move to the ignore class, and a spot check of
    one image against the oracle."""
    n, h, w = 6, 256, 480
    gen = torch.Generator(device=dev).manual_seed(3)
    mains, auxs = [], []
    for nm, c in SOURCES:
        m = 3 * torch.randn(n, c, h, w, generator=gen, device=dev)
        mains.append(m), auxs.append(m + 1.5 * torch.randn(n, c, h, w, generator=gen, device=dev))
    luts = [O.LUTS[nm] for nm, _ in SOURCES]
    for policy in ("all", "half"):
        r = ops.fuse_sources(mains, auxs, luts, policy=policy)
        ra = ops.fuse_sources([m[:3] for m in mains], [a[:3] for a in auxs], luts, policy=policy)
        rb = ops.fuse_sources([m[3:] for m in mains], [a[3:] for a in auxs], luts, policy=policy)
        assert torch.equal(torch.cat([ra.label, rb.label]), r.label)
        assert torch.equal(torch.cat([ra.conf, rb.conf]), r.conf) and torch.equal(torch.cat([ra.unc, rb.unc]), r.unc)
        assert torch.equal(ra.class_hist + rb.class_hist, r.class_hist)
        assert torch.equal(ra.conf_hist + rb.conf_hist, r.conf_hist)
        assert torch.equal(r.class_hist, torch.bincount(r.label.reshape(-1).long(), minlength=5))
        assert torch.equal(r.conf_hist.sum(dim=1), r.class_hist)
        assert int(r.class_hist.sum()) == n * h * w
        th, kept = ops.cb_thresholds(r.label, r.conf, 0.2, conf_hist=r.conf_hist.clone())
        # 2-way "sharded" thresholds: histograms of the two halves are summed before each select
        halves = [(ra.label, ra.conf), (rb.label, rb.conf)]
        th2 = _sharded_thresholds(ops, halves, 0.2)
        assert torch.equal(th, th2)
        th_ref, _ = O.cb_thresholds(r.label.cpu(), r.conf.cpu(), 0.2)
        assert torch.equal(th.cpu(), th_ref)
        final, mask, fh = ops.apply_thresholds(r.label, r.conf, th)
        assert bool(((final == r.label) | (final == 4)).all()) and torch.equal(mask == 1, final == 4)
        assert torch.equal(fh, torch.bincount(final.reshape(-1).long(), minlength=5))
        for k in range(1, 4):            # about `portion` of each class survives
            nk = int((r.label == k).sum())
            if nk > 100:
                assert abs(int((final == k).sum()) - int(nk * 0.2)) <= max(3, nk // 1000)
        ref = O.fuse_sources([m[:1].cpu() for m in mains], [a[:1].cpu() for a in auxs], luts, policy)
        assert not bool(((r.label[:1].cpu() != ref["label"]) & ~ref["marginal"]).any())
        torch.testing.assert_close(r.unc[:1].cpu(), ref["unc"], rtol=RTOL, atol=KLD_ATOL)


def _sharded_thresholds(ops, shards, portion):
    """Emulates N ranks on one GPU: per-pass histograms of all shards are summed (the all-reduce) before the select."""
    from mspl_b200 import _lib
    import ctypes
    lib = _lib.load()
    dev = shards[0][0].device
    K = 5
    state = torch.zeros(lib.mspl_radix_state_bytes(K), dtype=torch.uint8, device=dev)
    thresh = torch.empty(K, dtype=torch.float32, device=dev)
    hist = torch.zeros((K, 2048), dtype=torch.int64, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    for ps in range(3):
        for lab, conf in shards:
            hw = lab.shape[-1] * lab.shape[-2]
            _lib.check(lib.mspl_radix_hist_pass(p(lab), p(conf), lab.numel(), hw, K, ps, p(state), p(hist), 1, st), "hist")
        _lib.check(lib.mspl_radix_select(p(hist), K, ps, portion, p(state), p(thresh), None, st), "select")
    return thresh


def test_miou_matches_reference_golden(dev, golden):
    """GPU MIOU.get_iou against the live-reference fixture: integer areas, so exact."""
    from mspl_b200.utilities.metrics.segmentation_miou import MIOU
    g = golden("miou.npz")
    for nc in (5, 21):
        logits, target = _t(g["logits_%d" % nc]).to(dev), _t(g["target_%d" % nc]).to(dev)
        inter, union = MIOU(num_classes=nc).get_iou(logits, target)
        assert inter.dtype == np.float32 and union.dtype == np.float32
        assert np.array_equal(inter, g["inter_%d" % nc]) and np.array_equal(union, g["union_%d" % nc])
        inter, union = MIOU(num_classes=nc).get_iou((logits, logits), target)           # tuple outputs, as train() passes them
        assert np.array_equal(inter, g["inter_%d" % nc])
        pred = _t(g["pred_%d" % nc])
        for p in (pred.to(dev), pred.to(torch.uint8).to(dev)):
            inter, union = MIOU(num_classes=nc).get_iou(p, target)
            assert np.array_equal(inter, g["inter_lab_%d" % nc]) and np.array_equal(union, g["union_lab_%d" % nc])
    # full-size batch against the oracle (config 4 shape, one image)
    gen = torch.Generator().manual_seed(8)
    logits = torch.randn(2, 5, 256, 480, generator=gen)
    target = torch.randint(0, 6, (2, 256, 480), generator=gen)
    target[target == 5] = 255
    inter, union = MIOU(num_classes=5).get_iou(logits.to(dev), target.to(dev))
    i_ref, u_ref = O.miou_get_iou(logits, target, 5)
    assert np.array_equal(inter, i_ref) and np.array_equal(union, u_ref)


@pytest.mark.parametrize("num_sources,num_classes,src_classes,shape", [
    (1, 2, (3,), (2, 8, 16)),            # smallest supported K
    (5, 7, (37, 4, 9, 1, 20), (2, 24, 40)),   # K > 5 -> the 8-class instantiation; C not a multiple of the chunk; C = 1
    (8, 8, (6, 6, 6, 6, 6, 6, 6, 6), (1, 20, 36)),   # maximum S and K
    (2, 5, (256, 130), (1, 12, 20)),     # maximum source classes (uint8 argmax in the reference)
])
def test_generic_tables_sources_and_classes(ops, dev, num_sources, num_classes, src_classes, shape):
    """Arbitrary label tables, 1..8 sources, 2..8 target classes, 1..256 source classes, against the oracle."""
    n, h, w = shape
    gen = torch.Generator().manual_seed(num_sources * 100 + num_classes)
    mains, auxs, luts = [], [], []
    for s, c in enumerate(src_classes):
        m, a = O.synthetic_logits(n, c, h, w, seed=300 + s)
        mains.append(m), auxs.append(a)
        luts.append(torch.randint(0, num_classes, (c,), generator=gen).numpy())
    ignore = num_classes - 1
    for policy in ("half", "all", 1, "prob"):
        r = ops.fuse_sources([m.to(dev) for m in mains], [a.to(dev) for a in auxs], luts, policy=policy, num_classes=num_classes,
                             ignore_label=ignore, want_kld=True)
        ref = _oracle_generic(mains, auxs, luts, policy, num_classes, ignore)
        diff = r.label.cpu() != ref["label"]
        assert not bool((diff & ~ref["marginal"]).any())
        ok = ~diff
        torch.testing.assert_close(r.conf.cpu()[ok], ref["conf"][ok], rtol=RTOL, atol=1e-7)
        torch.testing.assert_close(r.unc.cpu(), ref["unc"], rtol=RTOL, atol=KLD_ATOL)
        if not bool(diff.any()):
            assert torch.equal(r.class_hist.cpu(), ref["class_hist"])
            th, kept = ops.cb_thresholds(r.label, r.conf, 0.3, num_classes=num_classes, conf_hist=r.conf_hist)
            th_ref, kept_ref = O.cb_thresholds(r.label.cpu(), r.conf.cpu(), 0.3, 1, num_classes)
            assert torch.equal(th.cpu(), th_ref) and torch.equal(kept.cpu(), kept_ref)


def _oracle_generic(mains, auxs, luts, policy, num_classes, ignore):
    """O.fuse_sources writes the reference's hard-coded ignore id 4 in merge_outputs; remap it for other class counts."""
    if ignore == 4:
        return O.fuse_sources(mains, auxs, luts, policy, num_classes, ignore)
    saved = O.IGNORE_LABEL
    O.IGNORE_LABEL = ignore
    try:
        return O.fuse_sources(mains, auxs, luts, policy, num_classes, ignore)
    finally:
        O.IGNORE_LABEL = saved


@pytest.mark.parametrize("out_size,main_size,aux_size", [((256, 480), (128, 240), (64, 120)),     # ESPDNetUE at the benchmark resolution
                                                         ((64, 96), (32, 48), (16, 24)),
                                                         ((48, 100), (24, 52), (12, 28)),          # non-integer scale factors
                                                         ((30, 44), (30, 44), (8, 12))])          # main already at full size
def test_fuse_sources_lowres(ops, dev, out_size, main_size, aux_size):
    """K1 with the network's final bilinear upsample fused in, against upsample-then-fuse on the CPU (its own parity
    definition, SURVEY.md 8f-1: the kernel and ATen's CPU interpolation round differently in the last ulp of a logit, which
    moves probabilities by up to ~1e-6, so labels are excused where the oracle's top-2 margin is below 1e-5 and floats get
    1e-4 relative / 1e-5 absolute)."""
    n = 2
    gen = torch.Generator().manual_seed(out_size[0])
    mains, auxs = [], []
    for nm, c in SOURCES:
        m = 3 * torch.randn(n, c, *main_size, generator=gen) + 3 * torch.randn(n, c, 1, 1, generator=gen)
        a = 3 * torch.randn(n, c, *aux_size, generator=gen)
        mains.append(m.contiguous()), auxs.append(a.contiguous())
    luts = [O.LUTS[nm] for nm, _ in SOURCES]
    saved = O.NEAR_TIE_MARGIN
    O.NEAR_TIE_MARGIN = 1e-5
    try:
        for policy in ("all", "half", "prob"):
            r = ops.fuse_sources_lowres([m.to(dev) for m in mains], [a.to(dev) for a in auxs], luts, out_size, policy=policy,
                                        want_kld=True)
            ref = O.fuse_sources_lowres(mains, auxs, luts, out_size, policy)
            diff = r.label.cpu() != ref["label"]
            assert not bool((diff & ~ref["marginal"]).any()), "%d mismatches outside near-ties" % int((diff & ~ref["marginal"]).sum())
            ok = ~diff
            torch.testing.assert_close(r.conf.cpu()[ok], ref["conf"][ok], rtol=1e-4, atol=1e-6)
            torch.testing.assert_close(r.unc.cpu(), ref["unc"], rtol=1e-4, atol=1e-5)
            for got, want in zip(r.kld, ref["kld"]):
                torch.testing.assert_close(got.cpu(), want, rtol=1e-4, atol=1e-5)
            assert torch.equal(r.class_hist, torch.bincount(r.label.reshape(-1).long(), minlength=5))
            assert torch.equal(r.conf_hist.sum(dim=1), r.class_hist)
            # and against the un-fused GPU path on GPU-upsampled logits: same labels except at near-ties
            ups = [O.upsample_heads(m.to(dev), a.to(dev), out_size) for m, a in zip(mains, auxs)]
            r2 = ops.fuse_sources([u[0].contiguous() for u in ups], [u[1].contiguous() for u in ups], luts, policy=policy)
            d2 = (r.label != r2.label).cpu()
            assert not bool((d2 & ~ref["marginal"]).any())
    finally:
        O.NEAR_TIE_MARGIN = saved


def test_labels_only_kernel(ops, dev, golden):
    """With no confidence / uncertainty / near-tie count requested under a vote policy the library runs its labels-only
    kernel (argmax of z, table, vote -- what the reference's loop keeps): identical labels and class counts."""
    g = golden("multi_source_3src.npz")
    mains, auxs, luts = _golden_sources(g)
    kw = dict(want_conf=False, want_unc=False, want_conf_hist=False, count_marginal=False)
    for policy in ("half", "all", 1, 2, 3):
        lean = _fuse(ops, dev, mains, auxs, luts, policy, **kw)
        full = _fuse(ops, dev, mains, auxs, luts, policy)
        assert lean.conf is None and lean.unc is None and lean.marginal is None
        assert torch.equal(lean.label, full.label) and torch.equal(lean.class_hist, full.class_hist)
        ref = O.fuse_sources(mains, auxs, luts, policy)
        assert not bool(((lean.label.cpu() != _t(g["label_%s" % policy])) & ~ref["marginal"]).any())
    # full-size images, partial tiles, 1..3 sources
    n, h, w = 3, 256, 480
    gen = torch.Generator(device=dev).manual_seed(4)
    big_m = [3 * torch.randn(n, c, h, w, generator=gen, device=dev) for _, c in SOURCES]
    big_a = [m + 1.5 * torch.randn(m.shape, generator=gen, device=dev) for m in big_m]
    for S in (1, 2, 3):
        for policy in ("half", "all"):
            lean = ops.fuse_sources(big_m[:S], big_a[:S], luts[:S], policy=policy, **kw)
            full = ops.fuse_sources(big_m[:S], big_a[:S], luts[:S], policy=policy)
            assert torch.equal(lean.label, full.label) and torch.equal(lean.class_hist, full.class_hist)


def test_vote_and_threshold_invariants(ops, dev):
    """Property tests (SURVEY.md section 4, T3): the voted label is always one some source proposed (or the ignore class),
    raising the vote threshold only ever turns labels into the ignore class, 'all' == int S, thresholds are monotone in the
    kept portion, and the label tables cover every source class."""
    n, h, w = 2, 64, 96
    mains, auxs = [], []
    for i, (nm, c) in enumerate(SOURCES):
        m, a = O.synthetic_logits(n, c, h, w, seed=500 + i)
        mains.append(m.to(dev)), auxs.append(a.to(dev))
    luts = [O.LUTS[nm] for nm, _ in SOURCES]
    for (nm, c) in SOURCES:
        assert len(O.LUTS[nm]) == c and set(np.unique(O.LUTS[nm])) <= {1, 2, 3, 4}      # no source class maps to 0
    per_source = []
    for m, a, lut in zip(mains, auxs, luts):
        z = m + 0.5 * a
        per_source.append(torch.as_tensor(lut, device=dev)[z.argmax(dim=1)])
    votes = torch.stack(per_source)                                                       # (S, n, h, w)
    labels = {t: ops.fuse_sources(mains, auxs, luts, policy=t).label.long() for t in (1, 2, 3)}
    assert torch.equal(labels[3], ops.fuse_sources(mains, auxs, luts, policy='all').label.long())
    assert torch.equal(labels[2], ops.fuse_sources(mains, auxs, luts, policy='half').label.long())
    for t, lab in labels.items():
        proposed = (votes == lab.unsqueeze(0)).any(dim=0)
        assert bool((proposed | (lab == 4)).all())
        agree = (votes == lab.unsqueeze(0)).sum(dim=0)
        assert bool(((agree >= t) | (lab == 4)).all())
    for lo, hi in ((1, 2), (2, 3)):
        changed = labels[lo] != labels[hi]
        assert bool((labels[hi][changed] == 4).all())
    r = ops.fuse_sources(mains, auxs, luts, policy='half')
    prev = None
    for p in (0.01, 0.1, 0.3, 0.7, 1.0):
        th, _ = ops.cb_thresholds(r.label, r.conf, p)
        if prev is not None:
            assert bool((th <= prev).all())
        prev = th
    # uncertainty is a mean of KL divergences: non-negative up to fp32 cancellation, and zero when the heads agree
    assert float(r.unc.min()) > -1e-5
    same = ops.fuse_sources(mains, [m.clone() for m in mains], luts, policy='half')
    assert float(same.unc.abs().max()) < 1e-5


def test_c_abi_error_codes(dev):
    """The C entry points validate their arguments and report through status codes (never a crash, never a launch)."""
    import ctypes
    from mspl_b200 import _lib
    lib = _lib.load()
    vp = ctypes.c_void_p
    m = torch.zeros(1, 5, 8, 8, device=dev)
    label = torch.zeros(1, 8, 8, dtype=torch.uint8, device=dev)
    hist = torch.zeros(5, dtype=torch.int64, device=dev)
    table = (ctypes.c_ubyte * 5)(3, 1, 1, 2, 2)
    ptrs = (vp * 1)(m.data_ptr())
    ncls = (ctypes.c_int * 1)(5)
    luts = (vp * 1)(ctypes.addressof(table))
    st = vp(torch.cuda.current_stream(dev).cuda_stream)

    def call(S=1, K=5, policy=0, ignore=4, ds=1, lab=label.data_ptr(), ch=hist.data_ptr(), cls=ncls, tab=luts):
        return lib.mspl_fuse_sources(S, ptrs, ptrs, cls, tab, 1, 64, K, policy, 1, ignore, ds, vp(lab), None, None, None, vp(ch),
                                     None, None, st)
    assert call() == 0
    assert call(S=0) == -1 and call(S=9) == -1 and call(K=1) == -1 and call(K=9) == -1
    assert call(policy=7) == -1 and call(ignore=5) == -1 and call(ds=0) == -1
    assert call(lab=0) == -1 and call(ch=0) == -1
    assert call(cls=(ctypes.c_int * 1)(0)) == -1 and call(cls=(ctypes.c_int * 1)(257)) == -1
    bad = (ctypes.c_ubyte * 5)(3, 1, 9, 2, 2)
    assert call(tab=(vp * 1)(ctypes.addressof(bad))) == -1                 # table value >= K
    assert call(ch=hist.data_ptr() + 4) == -2                               # misaligned histogram
    ws = torch.zeros(64, dtype=torch.uint8, device=dev)
    out3 = torch.zeros(3, device=dev)
    tgt = torch.zeros(1, 8, 8, dtype=torch.int64, device=dev)
    cw = torch.ones(5, device=dev)
    rc = lib.mspl_uw_ce_fwd_bwd(vp(m.data_ptr()), vp(m.data_ptr()), vp(tgt.data_ptr()), vp(cw.data_ptr()), 1, 5, 64, 20.0, 64.0, 1.0,
                                vp(out3.data_ptr()), None, None, vp(ws.data_ptr()), ws.numel(), st)
    assert rc == -5                                                          # workspace too small
    big = torch.zeros(lib.mspl_uw_ce_workspace_bytes(), dtype=torch.uint8, device=dev)
    m9 = torch.zeros(1, 9, 8, 8, device=dev)
    rc = lib.mspl_uw_ce_fwd_bwd(vp(m9.data_ptr()), vp(m9.data_ptr()), vp(tgt.data_ptr()), vp(cw.data_ptr()), 1, 9, 64, 20.0, 64.0, 1.0,
                                vp(out3.data_ptr()), None, None, vp(big.data_ptr()), big.numel(), st)
    assert rc == -3                                                          # more classes than the fused loss is built for
    assert lib.mspl_radix_select(None, 5, 0, 0.2, None, None, None, st) == -1
    assert lib.mspl_bracket_select(None, 5, 0.2, 4, None, None, None, None, None, None, st) == -1
    assert lib.mspl_cand_select(None, 5, 0, None, None, None, -1, st) == -1
    lab8 = torch.zeros(64, dtype=torch.uint8, device=dev)
    cf = torch.zeros(64, device=dev)
    br = torch.zeros(10, device=dev)
    cand = torch.zeros(64, dtype=torch.int32, device=dev)
    cnt = torch.zeros((), dtype=torch.int64, device=dev)
    # thresholds-only mode (ignore_label = -1) cannot write a label map
    assert lib.mspl_bracket_classify(vp(lab8.data_ptr()), vp(cf.data_ptr()), vp(br.data_ptr()), 64, 5, -1, vp(lab8.data_ptr()), None,
                                     None, vp(cand.data_ptr()), vp(cnt.data_ptr()), st) == -1
    assert lib.mspl_bracket_classify(vp(lab8.data_ptr()), vp(cf.data_ptr()), vp(br.data_ptr()), 2 ** 32, 5, 4, None, None, None,
                                     vp(cand.data_ptr()), vp(cnt.data_ptr()), st) == -3        # 32-bit candidate indices
    assert lib.mspl_conf_hist(vp(lab8.data_ptr()), vp(cf.data_ptr()), 64, 64, 9, vp(cnt.data_ptr()), 1, st) == -1
    torch.cuda.synchronize()


def test_non_contiguous_inputs_are_rejected(ops, dev):
    m = torch.zeros(2, 5, 8, 16, device=dev)
    with pytest.raises(ValueError, match="contiguous"):
        ops.fuse_sources([m[:, :, :, ::2]], [m[:, :, :, ::2]], [O.ID_FOREST_TO_GREENHOUSE])
    with pytest.raises(ValueError):
        ops.fuse_sources([m], [m[:1]], [O.ID_FOREST_TO_GREENHOUSE])
    with pytest.raises(ValueError):
        ops.fuse_sources([m.double()], [m.double()], [O.ID_FOREST_TO_GREENHOUSE])


def test_tma_and_scalar_kernels_agree_bitwise_at_scale(ops, dev):
    """The TMA-staged kernel (aligned tensors) and the scalar fallback kernel (the same data behind a 4-byte-offset view) run
    the identical per-pixel arithmetic, so a large batch must come out bit-for-bit equal -- a race or a mis-staged tile in
    the asynchronous pipeline would show up here long before it shows up on the small oracle-sized cases."""
    n, h, w = 48, 256, 480
    gen = torch.Generator(device=dev).manual_seed(77)
    mains, auxs, mains_off, auxs_off = [], [], [], []
    for nm, c in SOURCES:
        cnt = n * c * h * w
        bm = torch.empty(cnt + 1, device=dev).normal_(0, 3, generator=gen)
        ba = torch.empty(cnt + 1, device=dev).normal_(0, 3, generator=gen)
        mains_off.append(bm[1:].view(n, c, h, w)), auxs_off.append(ba[1:].view(n, c, h, w))        # 4-byte aligned only
        mains.append(bm[1:].clone().view(n, c, h, w)), auxs.append(ba[1:].clone().view(n, c, h, w))   # 16-byte aligned copies
    luts = [O.LUTS[nm] for nm, _ in SOURCES]
    for policy in ("all", "half", "prob"):
        a = ops.fuse_sources(mains, auxs, luts, policy=policy, want_kld=True)
        b = ops.fuse_sources(mains_off, auxs_off, luts, policy=policy, want_kld=True)
        assert torch.equal(a.label, b.label) and torch.equal(a.conf, b.conf) and torch.equal(a.unc, b.unc)
        assert all(torch.equal(x, y) for x, y in zip(a.kld, b.kld))
        assert torch.equal(a.class_hist, b.class_hist) and torch.equal(a.conf_hist, b.conf_hist)
        assert int(a.marginal) == int(b.marginal)
        # and run-to-run determinism of the asynchronous pipeline
        a2 = ops.fuse_sources(mains, auxs, luts, policy=policy)
        assert torch.equal(a.label, a2.label) and torch.equal(a.conf, a2.conf) and torch.equal(a.unc, a2.unc)


@pytest.mark.parametrize("tag", ["hard", "soft", "bins8"])
def test_nid_loss_matches_reference_golden(dev, golden, tag):
    """NIDLoss forward and backward against the live-reference fixture (loss within 1e-4 absolute -- it is (NID - 0.95) * 20,
    a difference of O(1) quantities; gradients 1e-3 relative with a 1e-4 * max|grad| floor: they pass through
    sigmoid(x / bw) windows with bw down to 1e-3, i.e. slopes of 1e3, in fp32)."""
    from mspl_b200.loss_fns.segmentation_loss import NIDLoss
    g = golden("nid.npz")
    k, lb, bwc, bwl = g["cfg_" + tag]
    crit = NIDLoss(image_bin=int(k), label_bin=int(lb), bw_camera=float(bwc), bw_label=float(bwl))
    camera = _t(g["camera_" + tag]).to(dev)
    label = _t(g["label_" + tag]).to(dev).requires_grad_(True)
    loss = crit(camera, label)
    loss.backward()
    assert abs(loss.item() - float(g["loss_" + tag])) <= 1e-4
    want = _t(g["grad_" + tag])
    scale = float(want.abs().max())
    if scale == 0.0:
        assert float(label.grad.abs().max()) < 1e-6
    else:
        torch.testing.assert_close(label.grad.cpu(), want, rtol=1e-3, atol=1e-4 * scale)
    # an upstream gradient is applied on the device
    label2 = _t(g["label_" + tag]).to(dev).requires_grad_(True)
    (crit(camera, label2) * 0.5).backward()
    torch.testing.assert_close(label2.grad, label.grad * 0.5, rtol=1e-6, atol=0)


def test_nid_loss_full_size_vs_oracle(dev):
    from mspl_b200.loss_fns.segmentation_loss import NIDLoss
    gen = torch.Generator().manual_seed(6)
    camera = torch.rand(4, 3, 64, 96, generator=gen)
    label = 0.004 * torch.randn(4, 5, 64, 96, generator=gen)
    lab = label.clone().requires_grad_(True)
    want = O.nid_loss(camera, lab, 16, 5, 0.005, 0.05)
    gw, = torch.autograd.grad(want, lab)
    ld = label.to(dev).requires_grad_(True)
    got = NIDLoss(16, 5, 0.005, 0.05)(camera.to(dev), ld)
    got.backward()
    assert abs(got.item() - want.item()) <= 1e-4
    torch.testing.assert_close(ld.grad.cpu(), gw, rtol=1e-3, atol=1e-4 * float(gw.abs().max()))


def test_in_training_visualization_matches_reference_golden(dev, golden):
    """The TensorBoard hook (utilities/utils.py:76-133) with the maps computed on the device: same tags in the same order,
    identical image / label grids, KLD heat map within 1e-5."""
    from collections import OrderedDict
    from oracle.make_golden import GREENHOUSE_ENCODING, CapturingWriter
    from mspl_b200.utilities.utils import in_training_visualization_img, prediction_maps
    g = golden("visualization.npz")
    images, main, aux, labels = (_t(g[k]).to(dev) for k in ("images", "main", "aux", "labels"))
    enc = OrderedDict(GREENHOUSE_ENCODING)
    wr = CapturingWriter()
    in_training_visualization_img(None, images, labels=labels, predictions=(main, aux), class_encoding=enc, writer=wr, epoch=0,
                                  data='train')
    assert wr.order == list(g["tuple_order"])
    assert np.array_equal(wr.images["train/images"], g["tuple_train_images"])
    assert np.array_equal(wr.images["train/train_labels"], g["tuple_train_train_labels"])
    assert np.array_equal(wr.images["train/pred_labels"], g["tuple_train_pred_labels"])
    np.testing.assert_allclose(wr.images["train/kld"], g["tuple_train_kld"], rtol=0, atol=1e-5)
    wr = CapturingWriter()
    in_training_visualization_img(None, images, labels=None, predictions=main, class_encoding=enc, writer=wr, epoch=0, data='val')
    assert wr.order == list(g["tensor_order"])
    assert np.array_equal(wr.images["val/pred_labels"], g["tensor_val_pred_labels"])
    # OrderedDict predictions (torchvision-style heads) and a model call
    pred_od, heat_od = prediction_maps(OrderedDict([('out', main), ('aux', aux)]))
    pred_t, heat_t = prediction_maps((main, aux))
    assert torch.equal(pred_od, pred_t) and torch.equal(heat_od, heat_t)
    ref_pred, ref_heat = O.visualization_maps(main.cpu(), aux.cpu())
    assert torch.equal(pred_t.cpu(), ref_pred)
    torch.testing.assert_close(heat_t.cpu(), ref_heat, rtol=0, atol=1e-5)

    class Net(torch.nn.Module):
        def forward(self, x):
            return main, aux
    wr = CapturingWriter()
    in_training_visualization_img(Net(), images, labels=labels, class_encoding=enc, writer=wr, epoch=1, data='train')
    assert np.array_equal(wr.images["train/pred_labels"], g["tuple_train_pred_labels"])
    # exact ties -> first maximal index; labels outside the colour table -> black
    tied = torch.zeros(1, 5, 4, 8, device=dev)
    p, _ = prediction_maps(tied)
    assert int(p.abs().sum()) == 0
    from mspl_b200 import ops
    rgb = ops.label_colors(torch.tensor([[[0, 4, 7, -1]]], device=dev), [c for _, c in GREENHOUSE_ENCODING])
    assert rgb[0, :, 0, 0].tolist() == [0, 255, 0] and rgb[0, :, 0, 2].tolist() == [0, 0, 0] and rgb[0, :, 0, 3].tolist() == [0, 0, 0]
