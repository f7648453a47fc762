"""Pins the oracle against the LIVE reference (only where /root/reference exists, i.e. the build
container; skipped on the GPU box).  Fresh seeds, so this is independent of the golden fixtures."""
import numpy as np
import pytest
import torch

from oracle import mspl_oracle as O
from oracle.ref_import import FixedLogitsModel, build_espdnetue, load_reference, reference_available

pytestmark = pytest.mark.skipif(not reference_available(), reason="reference tree not present")

SOURCES = (("camvid", 13), ("cityscapes", 20), ("forest", 5))


@pytest.fixture(scope="module")
def ref():
    r = load_reference()
    yield r
    torch.autograd.set_detect_anomaly(False)   # the reference loss switches it on globally


def _close(a, b, rtol=4e-7, atol=4e-7):
    np.testing.assert_allclose(np.asarray(a), np.asarray(b), rtol=rtol, atol=atol)


def test_luts(ref):
    for name, _ in SOURCES:
        assert np.array_equal(getattr(ref.greenhouse, "id_%s_to_greenhouse" % name), O.LUTS[name])


@pytest.mark.parametrize("policy", [None, "half", "all", 1, 2, 3, "3", 7, True, False])
def test_label_generation_matches_reference(ref, policy):
    gen = torch.Generator().manual_seed(11)
    n, h, w = 2, 20, 36
    mains, auxs = [], []
    for _, c in SOURCES:
        m = 3 * torch.randn(n, c, h, w, generator=gen)
        mains.append(m), auxs.append(m + 1.5 * torch.randn(n, c, h, w, generator=gen))
    luts = [O.LUTS[s] for s, _ in SOURCES]
    got, got_ca = O.multi_source_labels(mains, auxs, luts, policy)
    for i in range(n):
        per = []
        for (name, _), m, a in zip(SOURCES, mains, auxs):
            out, kld = ref.uest.get_output(FixedLogitsModel(m[i:i + 1], a[i:i + 1]), torch.zeros(1), device='cpu')
            o2, k2 = O.get_output_from_logits(m[i:i + 1], a[i:i + 1])
            _close(o2, out, atol=0), _close(k2, kld)
            amax = np.asarray(np.argmax(out.transpose(1, 2, 0), axis=2), dtype=np.uint8)
            lab_s = getattr(ref.greenhouse, "id_%s_to_greenhouse" % name)[amax]
            assert np.array_equal(lab_s, O.argmax_to_greenhouse(o2, O.LUTS[name]))
            assert np.array_equal(ref.uest.transfer_id_to_greenhouse(O.LUTS[name], amax), lab_s)
            per.append(lab_s)
        want = ref.uest.merge_outputs(np.array(per), seg_classes=5, thresh=policy)
        assert want.dtype == np.int64
        assert np.array_equal(got[i], want)
        assert np.array_equal(O.merge_outputs(np.array(per), 5, policy), want)


def test_loss_matches_reference(ref):
    gen = torch.Generator().manual_seed(5)
    b, k, h, w = 3, 5, 12, 20
    main = 2 * torch.randn(b, k, h, w, generator=gen)
    aux = main + torch.randn(b, k, h, w, generator=gen)
    target = torch.randint(0, k, (b, h, w), generator=gen)
    cw = torch.tensor([0.0, 2.0, 5.0, 1.5, 9.0])
    crit = ref.seg_loss.UncertaintyWeightedSegmentationLoss(k, class_weights=cw.clone(), ignore_idx=4, device='cpu')
    m, a = main.clone().requires_grad_(True), aux.clone().requires_grad_(True)
    kld = ref.seg_loss.PixelwiseKLD()(m, a)
    loss = crit(m + 0.5 * a, target, kld) * 20 + kld.mean()
    gm, ga = torch.autograd.grad(loss, (m, a))
    w_o = O.make_class_weights(k, cw.clone(), 4)
    assert torch.equal(w_o, crit.class_weights)
    l_o, gm_o, ga_o = O.training_loss_and_grads(main, aux, target, w_o)
    _close(l_o, loss.detach(), rtol=1e-6), _close(gm_o, gm, rtol=1e-6, atol=1e-10), _close(ga_o, ga, rtol=1e-6, atol=1e-10)
    # closed-form gradients used by the fused kernel (SURVEY.md 8a) against reference autograd in fp64
    l64, gm64, ga64 = O.training_loss_and_grads(main, aux, target, w_o, dtype=torch.float64)
    m64, a64 = main.double().requires_grad_(True), aux.double().requires_grad_(True)
    crit64 = ref.seg_loss.UncertaintyWeightedSegmentationLoss(k, class_weights=w_o.double(), ignore_idx=4, device='cpu')
    kld64 = ref.seg_loss.PixelwiseKLD()(m64, a64)
    loss64 = crit64(m64 + 0.5 * a64, target, kld64) * 20 + kld64.mean()
    g1, g2 = torch.autograd.grad(loss64, (m64, a64))
    _close(l64, loss64.detach(), rtol=1e-13, atol=0), _close(gm64, g1, rtol=1e-12, atol=1e-18), _close(ga64, g2, rtol=1e-12, atol=1e-18)


def test_config1_full_resolution(ref):
    """BASELINE config 1 (two of its eight images here to keep the CPU suite short): random-init 20-class
    ESPDNetUE at 256x480, reference CPU path vs the oracle on the very same logits."""
    model = build_espdnetue(20, seed=3)
    gen = torch.Generator().manual_seed(3)
    lut = ref.greenhouse.id_cityscapes_to_greenhouse
    with torch.no_grad():
        for _ in range(2):
            image = torch.randn(1, 3, 256, 480, generator=gen)
            main, aux = model(image)
            out, kld = ref.uest.get_output(model, image, device='cpu')
            o2, k2 = O.get_output_from_logits(main, aux)
            _close(o2, out, atol=0), _close(k2, kld)
            amax = np.asarray(np.argmax(out.transpose(1, 2, 0), axis=2), dtype=np.uint8)
            want = ref.uest.merge_outputs(np.array([lut[amax]]), seg_classes=5, thresh=None)
            got, _ = O.multi_source_labels([main], [aux], [O.ID_CITYSCAPES_TO_GREENHOUSE], None)
            assert np.array_equal(got[0], want)


def test_miou_matches_reference(ref):
    import sys
    from utilities.metrics.segmentation_miou import MIOU
    gen = torch.Generator().manual_seed(17)
    for nc in (5, 21):
        logits = torch.randn(2, nc, 18, 26, generator=gen)
        target = torch.randint(0, nc + 2, (2, 18, 26), generator=gen)
        target[target == nc + 1] = 255
        want = MIOU(num_classes=nc).get_iou(logits.clone(), target.clone())
        got = O.miou_get_iou(logits, target, nc)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_nid_loss_matches_reference(ref):
    orig_to = torch.Tensor.to

    def to_cpu(self, *a, **k):       # the reference hard-codes .to('cuda')
        a = tuple('cpu' if (isinstance(x, str) and x.startswith('cuda')) else x for x in a)
        return orig_to(self, *a, **k)
    torch.Tensor.to = to_cpu
    try:
        gen = torch.Generator().manual_seed(23)
        camera = torch.rand(2, 3, 10, 14, generator=gen)
        label = 0.004 * torch.randn(2, 5, 10, 14, generator=gen)
        a = label.clone().requires_grad_(True)
        want = ref.seg_loss.NIDLoss(image_bin=16, label_bin=5, bw_label=0.05)(camera, a)
        gw, = torch.autograd.grad(want, a)
    finally:
        torch.Tensor.to = orig_to
    b = label.clone().requires_grad_(True)
    got = O.nid_loss(camera, b, 16, 5, 0.005, 0.05)
    gg, = torch.autograd.grad(got, b)
    _close(got.detach(), want.detach(), rtol=1e-6, atol=1e-6)
    _close(gg, gw, rtol=1e-5, atol=1e-6)


def _sweep_cases(count, seed):
    import random
    rng = random.Random(seed)
    out = []
    for i in range(count):
        srcs = rng.sample(SOURCES, rng.choice([1, 2, 3]))
        out.append((i, srcs, rng.choice([(1, 7, 9), (2, 16, 24), (1, 1, 40), (3, 12, 5)]), rng.choice([0.05, 1.0, 3.0, 12.0, 40.0]),
                    rng.random() < 0.3, rng.choice([None, "half", "all", 1, 2, 3])))
    return out


@pytest.mark.parametrize("case", _sweep_cases(24, seed=606), ids=lambda c: "ref%02d" % c[0])
def test_oracle_sweep_against_live_reference(ref, case):
    """Seeded sweep of the oracle against the LIVE reference: source subsets and orders, shapes, logit scales from 0.05 to 40,
    quantised logits (exact ties -> first-index rules of np.argmax / merge_outputs), every vote policy; then the loss and the
    training loop's metric statements on the same tensors."""
    i, srcs, (n, h, w), sigma, ties, policy = case
    gen = torch.Generator().manual_seed(7000 + i)
    mains, auxs = [], []
    for _, c in srcs:
        m = sigma * torch.randn(n, c, h, w, generator=gen)
        a = m + 0.5 * sigma * torch.randn(n, c, h, w, generator=gen)
        if ties:
            m, a = torch.round(m), torch.round(2 * a) / 2
        mains.append(m), auxs.append(a)
    luts = [O.LUTS[s] for s, _ in srcs]
    got, got_ca = O.multi_source_labels(mains, auxs, luts, policy)
    want_ca = np.zeros(5)
    for j in range(n):
        per = []
        for (name, _), m, a in zip(srcs, mains, auxs):
            out, kld = ref.uest.get_output(FixedLogitsModel(m[j:j + 1], a[j:j + 1]), torch.zeros(1), device='cpu')
            o2, k2 = O.get_output_from_logits(m[j:j + 1], a[j:j + 1])
            _close(o2, out, atol=0)
            _close(k2, kld, rtol=1e-6, atol=4e-7 * max(1.0, sigma))
            amax = np.asarray(np.argmax(out.transpose(1, 2, 0), axis=2), dtype=np.uint8)
            per.append(getattr(ref.greenhouse, "id_%s_to_greenhouse" % name)[amax])
        want = ref.uest.merge_outputs(np.array(per), seg_classes=5, thresh=policy)
        assert np.array_equal(got[j], want)
        for k in range(5):                                      # class_array as the loop accumulates it (:919-921)
            want_ca[k] += (want == k).sum()
    assert np.array_equal(got_ca, want_ca)

    # loss + metric on the first source's first five classes
    k = min(5, mains[0].shape[1])
    main, aux = mains[0][:, :k].contiguous(), auxs[0][:, :k].contiguous()
    target = torch.randint(0, k, (n, h, w), generator=gen)
    cw = torch.rand(k, generator=gen) * 3
    crit = ref.seg_loss.UncertaintyWeightedSegmentationLoss(k, class_weights=cw.clone(), ignore_idx=k - 1, device='cpu')
    m, a = main.clone().requires_grad_(True), aux.clone().requires_grad_(True)
    kld = ref.seg_loss.PixelwiseKLD()(m, a)
    loss = crit(m + 0.5 * a, target, kld) * 20 + kld.mean()
    gm, ga = torch.autograd.grad(loss, (m, a))
    l_o, gm_o, ga_o = O.training_loss_and_grads(main, aux, target, O.make_class_weights(k, cw.clone(), k - 1))
    _close(l_o, loss.detach(), rtol=1e-6, atol=1e-12)
    _close(gm_o, gm, rtol=1e-6, atol=1e-10), _close(ga_o, ga, rtol=1e-6, atol=1e-10)
    from utilities.metrics.segmentation_miou import MIOU
    tgt = target.clone()
    tgt[0, 0, :2] = 255
    inter, union = MIOU(num_classes=k).get_iou(main, tgt) if k > 1 else (None, None)
    if k > 1:
        i_o, u_o = O.miou_get_iou(main, tgt, num_classes=k)
        assert np.array_equal(i_o, inter) and np.array_equal(u_o, union)
