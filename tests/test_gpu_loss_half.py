"""K4 on fp16 / bf16 logits (mixed-precision training): the explicit form against the fp32 kernel on the upcast logits and
against the fp64 oracle, the deferred autograd form and its loss scaling, a training step under torch.autocast, and the
inputs that are still refused."""
import os
import sys

import pytest
import torch

from oracle import mspl_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gpu_launch_probe import dev, launches, ops  # noqa: E402,F401

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
SCALES = [1.0, 0.25, 3.0, 2.0 ** 16]


def _logits(n, k, h, w, dtype, device, seed, offset=0):
    """Correlated main / aux heads rounded to `dtype`; offset > 0 places each tensor `offset` elements into its buffer, so the
    planes are only 2-byte aligned and K4 falls back to one pixel per thread."""
    m, a = O.synthetic_logits(n, k, h, w, seed=seed)
    out = []
    for x in (m, a):
        buf = torch.empty(x.numel() + offset, dtype=dtype, device=device)
        v = buf[offset:].view(x.shape)
        v.copy_(x.to(dtype))
        out.append(v)
    return out


def _targets(n, k, h, w, u8, device, seed, invalid=True):
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(0, k, (n, h, w), generator=g)
    if invalid:
        t[torch.rand((n, h, w), generator=g) < 0.05] = 255          # outside [0, K): contributes like a zero-weight class
    return t.to(torch.uint8 if u8 else torch.int64).to(device)


def _ordered(x):
    """Signed-magnitude bit pattern of a 2-byte float as a monotone integer (+0 and -0 both 0): neighbours differ by 1."""
    b = x.contiguous().view(torch.int16).to(torch.int32)
    return torch.where(b < 0, -(b & 0x7fff), b)


def _within_one_ulp(got, want, what):
    """Rule of this file: every element within one unit in the last place of `want`, at least 99.9 % bit-equal.  (The vector
    widths of the two kernels may differ, and with them the contraction of multiply-adds, test_fused_loss_uint8_targets.)"""
    assert got.dtype == want.dtype and got.shape == want.shape
    d = (_ordered(got) - _ordered(want)).abs()
    assert int(d.max()) <= 1, "%s: %d ulp apart" % (what, int(d.max()))
    assert float((d == 0).float().mean()) >= 0.999, "%s: only %.4f bit-equal" % (what, float((d == 0).float().mean()))


def _cw(k, device):
    w = torch.linspace(0.5, 1.5, k)
    if k > 1:
        w[-1] = 0.0
    return w.to(device)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("k", [1, 2, 5, 8])
def test_half_matches_fp32_kernel_on_upcast_logits(ops, dev, dtype, u8, k):
    """The fp16 / bf16 instantiations compute what the fp32 kernel computes on main.float(), aux.float(): equal IoU counts,
    out3 to 1e-6 (the summation order follows the vector width and the grid), gradients under the one-ulp rule, with the scale
    given on the host or as the device scalar.  Rows of 8-pixel multiples, an odd width, and 2-byte aligned planes."""
    cw = _cw(k, dev)
    for shape, offset in (((2, 24, 40), 0), ((3, 7, 13), 0), ((2, 16, 40), 1)):
        n, h, w = shape
        main, aux = _logits(n, k, h, w, dtype, dev, seed=100 + k, offset=offset)
        tgt = _targets(n, k, h, w, u8, dev, seed=7 + k)
        m32, a32 = main.float(), aux.float()
        for iou in (False, True):
            cnt_h = torch.zeros((3, k), dtype=torch.int64, device=dev) if iou else None
            cnt_f = torch.zeros((3, k), dtype=torch.int64, device=dev) if iou else None
            o_h, dm, da = ops.uw_ce_fwd_bwd(main, aux, tgt, cw, backward=False, iou_counts=cnt_h)
            o_f, _, _ = ops.uw_ce_fwd_bwd(m32, a32, tgt, cw, backward=False, iou_counts=cnt_f)
            assert dm is None and da is None and o_h.dtype == torch.float32
            torch.testing.assert_close(o_h, o_f, rtol=1e-6, atol=0)
            if iou:
                assert torch.equal(cnt_h, cnt_f)
            for s in SCALES:
                _, g32m, g32a = ops.uw_ce_fwd_bwd(m32, a32, tgt, cw, grad_scale=s)
                want_m, want_a = g32m.to(dtype), g32a.to(dtype)
                sd = torch.tensor([s], dtype=torch.float32, device=dev)
                for kw in (dict(grad_scale=s), dict(grad_scale_dev=sd)):
                    if iou:
                        cnt_h.zero_()
                        cnt_f.zero_()
                        ops.uw_ce_fwd_bwd(m32, a32, tgt, cw, backward=False, iou_counts=cnt_f)
                    o_h, dm, da = ops.uw_ce_fwd_bwd(main, aux, tgt, cw, iou_counts=cnt_h, **kw)
                    assert dm.dtype == dtype and da.dtype == dtype
                    torch.testing.assert_close(o_h, o_f, rtol=1e-6, atol=0)
                    if iou:
                        assert torch.equal(cnt_h, cnt_f)
                    what = "%s %s K=%d %s offset=%d %s" % (dtype, "u8" if u8 else "i64", k, shape, offset, kw)
                    _within_one_ulp(dm, want_m, "d_main " + what)
                    _within_one_ulp(da, want_a, "d_aux " + what)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("u8", [False, True])
def test_half_matches_fp64_oracle(ops, dev, dtype, u8):
    """Against the fp64 restated forward on the upcast logits: loss to 1e-5; gradients to the dtype's unit roundoff
    (2^-8 bf16, 2^-11 fp16: the rounding of the result) plus 1e-4 relative for the fp32 arithmetic, with an absolute floor of
    1e-5 of max |grad| and half the smallest subnormal (values below fp16's normal range keep fewer bits)."""
    n, k, h, w = 2, 5, 32, 48
    main, aux = _logits(n, k, h, w, dtype, dev, seed=21)
    tgt = _targets(n, k, h, w, u8, dev, seed=22, invalid=False)
    cw = torch.tensor([1.0, 0.7, 1.3, 1.0, 0.0])
    l64, gm64, ga64 = O.training_loss_and_grads(main.cpu().double(), aux.cpu().double(), tgt.cpu().long(), cw.double(),
                                                dtype=torch.float64)
    u = 2.0 ** -8 if dtype == torch.bfloat16 else 2.0 ** -11
    sub = 2.0 ** -134 if dtype == torch.bfloat16 else 2.0 ** -25
    for s in (1.0, 2.0 ** 16):
        out3, dm, da = ops.uw_ce_fwd_bwd(main, aux, tgt, cw.to(dev), grad_scale=s)
        assert abs(out3[0].item() - l64.item()) <= 1e-5 * abs(l64.item())
        for got, ref in ((dm, gm64), (da, ga64)):
            ref = ref * s
            err = (got.cpu().double() - ref).abs()
            tol = (u + 1e-4) * ref.abs() + max(1e-5 * float(ref.abs().max()), sub)
            assert bool((err <= tol).all()), "max excess %.3g" % float((err - tol).max())


@pytest.mark.parametrize("dtype", DTYPES)
def test_autograd_half_equals_explicit_form(ops, dev, dtype):
    """FusedUncertaintyWeightedLoss on fp16 / bf16 leaves: .grad in the leaves' dtype, equal to the explicit one-launch form
    with the same upstream scale (same instantiation, same scale value: bit-equal), the IoU counts of the forward launch."""
    from mspl_b200.loss_fns.segmentation_loss import FusedUncertaintyWeightedLoss
    n, k, h, w = 2, 5, 32, 64
    main, aux = _logits(n, k, h, w, dtype, dev, seed=31)
    tgt = _targets(n, k, h, w, True, dev, seed=32)
    crit = FusedUncertaintyWeightedLoss(k, _cw(k, dev).clone(), track_iou=True)
    for s in (1.0, 3.0, 2.0 ** 16):
        crit.reset_iou()
        m, a = main.clone().requires_grad_(True), aux.clone().requires_grad_(True)
        loss = crit(m, a, tgt)
        (loss * s).backward()
        out3, dm, da = ops.uw_ce_fwd_bwd(main, aux, tgt, crit.class_weights, grad_scale=s)
        assert m.grad.dtype == dtype and a.grad.dtype == dtype
        assert torch.equal(m.grad, dm) and torch.equal(a.grad, da)
        assert torch.equal(crit.last_parts, out3) and loss.dtype == torch.float32
        cnt = torch.zeros((3, k), dtype=torch.int64, device=dev)
        ops.uw_ce_fwd_bwd(main.float(), aux.float(), tgt, crit.class_weights, backward=False, iou_counts=cnt)
        assert torch.equal(crit.iou_counts, cnt)


def test_grad_scaler_scales_before_rounding(ops, dev):
    """B = 8 x 256 x 480 fp16 logits under torch.amp.GradScaler (initial scale 2^16): the gradients are round_fp16(s * g32)
    under the one-ulp rule.  Rounding first and scaling afterwards, round_fp16(g32) * s, would zero more than 5 % of the
    elements that are non-zero here."""
    n, k, h, w = 8, 5, 256, 480
    main, aux = _logits(n, k, h, w, torch.float16, dev, seed=41)
    tgt = _targets(n, k, h, w, True, dev, seed=42)
    cw = _cw(k, dev)
    scaler = torch.amp.GradScaler("cuda")
    m, a = main.clone().requires_grad_(True), aux.clone().requires_grad_(True)
    loss = ops.uw_ce_loss(m, a, tgt, cw)
    scaler.scale(loss).backward()
    s = float(scaler.get_scale())
    assert s == 2.0 ** 16
    _, g32m, g32a = ops.uw_ce_fwd_bwd(main.float(), aux.float(), tgt, cw)
    for got, g32, nm in ((m.grad, g32m, "d_main"), (a.grad, g32a, "d_aux")):
        _within_one_ulp(got, (g32 * s).half(), nm)
        nonzero = got != 0
        lost = nonzero & (g32.half() == 0)
        share = float(lost.sum()) / float(nonzero.sum())
        print("%s: rounding before scaling would zero %.1f %% of the non-zero gradients" % (nm, 100 * share))
        assert share > 0.05


@pytest.mark.parametrize("dtype", DTYPES)
def test_one_launch_per_direction(ops, dev, launches, dtype):
    """torch.profiler: the forward runs K4 once (forward-only instantiation), the backward runs it once (forward+backward),
    and neither launches a cast, copy or scale kernel."""
    n, k, h, w = 4, 5, 64, 96
    main, aux = _logits(n, k, h, w, dtype, dev, seed=51)
    tgt = _targets(n, k, h, w, True, dev, seed=52)
    m, a = main.clone().requires_grad_(True), aux.clone().requires_grad_(True)
    cw = _cw(k, dev)
    ops.uw_ce_loss(m, a, tgt, cw).backward()           # warm-up: workspace, modules
    m.grad = a.grad = None

    def check(ks, bwd):
        k4 = [x for x in ks if "uw_ce_fused_half_kernel" in x.name]
        assert len(k4) == 1 and (",%s,unsignedchar,false," % str(bwd).lower()) in k4[0].name, [x.name[:90] for x in ks]
        bad = [x.name[:90] for x in ks if any(f in x.name.lower() for f in ("copy", "cast", "convert", "scale_inplace"))]
        assert not bad, bad
    loss, ks = launches(lambda: ops.uw_ce_loss(m, a, tgt, cw))
    check(ks, False)
    _, ks = launches(lambda: loss.backward())
    check(ks, True)
    assert m.grad.dtype == dtype


class _TwoLayerNet(torch.nn.Module):
    def __init__(self, k):
        super().__init__()
        self.c1 = torch.nn.Conv2d(3, 16, 3, padding=1)
        self.c2 = torch.nn.Conv2d(16, 2 * k, 1)
        self.k = k

    def forward(self, x):
        y = self.c2(torch.relu(self.c1(x)))
        return y[:, :self.k], y[:, self.k:]


def _step(net, images, labels, loss_fn, cast):
    net.zero_grad(set_to_none=True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        pred, pred_aux = net(images)
        assert pred.dtype == torch.bfloat16
        if cast:
            pred, pred_aux = pred.float(), pred_aux.float()
        loss = loss_fn(pred, pred_aux, labels)
    loss.backward()
    return loss.detach(), [p.grad.clone() for p in net.parameters()]


def _close(got, want, rtol, what):
    rel = float((got.float() - want.float()).norm() / want.float().norm().clamp_min(1e-30))
    assert rel <= rtol, "%s: relative error %.3g > %.3g" % (what, rel, rtol)


def test_training_step_under_autocast(ops, dev):
    """A two-layer conv net trained one step under torch.autocast(bf16), with the reference-shaped expression and with the
    fused module, against the same step with the logits cast to fp32 before the loss.  Fused: the kernel sees the same
    (upcast) values, so the loss agrees to 1e-5 and the parameter gradients, which differ only by the one-ulp rule on the logit
    gradients, to 1e-2 in norm; the IoU counts are equal.  Reference expression: `pred + 0.5 * pred_aux` is itself rounded
    to bf16 under autocast, so loss and gradients agree to 2e-2."""
    from mspl_b200.loss_fns.segmentation_loss import (FusedUncertaintyWeightedLoss, PixelwiseKLD,
                                                      UncertaintyWeightedSegmentationLoss)
    torch.manual_seed(0)
    k = 5
    net = _TwoLayerNet(k).to(dev)
    g = torch.Generator().manual_seed(61)
    images = torch.randn((2, 3, 64, 96), generator=g).to(dev)
    labels = torch.randint(0, k, (2, 64, 96), generator=g).to(dev)
    cw = torch.ones(k, device=dev)
    criterion = UncertaintyWeightedSegmentationLoss(k, cw.clone(), ignore_idx=4)
    kld_mod = PixelwiseKLD()

    def reference(pred, pred_aux, lab):
        kld = kld_mod(pred, pred_aux)
        return criterion(pred + 0.5 * pred_aux, lab, kld) * 20 + kld.mean()
    l_h, g_h = _step(net, images, labels, reference, cast=False)
    l_f, g_f = _step(net, images, labels, reference, cast=True)
    assert l_h.dtype == torch.float32
    _close(l_h, l_f, 2e-2, "reference-shaped loss")
    for i, (a, b) in enumerate(zip(g_h, g_f)):
        _close(a, b, 2e-2, "reference-shaped grad %d" % i)

    fused_h = FusedUncertaintyWeightedLoss(k, cw.clone(), ignore_idx=4, track_iou=True)
    fused_f = FusedUncertaintyWeightedLoss(k, cw.clone(), ignore_idx=4, track_iou=True)
    l_h, g_h = _step(net, images, labels, fused_h, cast=False)
    l_f, g_f = _step(net, images, labels, fused_f, cast=True)
    _close(l_h, l_f, 1e-5, "fused loss")
    for i, (a, b) in enumerate(zip(g_h, g_f)):
        _close(a, b, 1e-2, "fused grad %d" % i)
    assert torch.equal(fused_h.iou_counts, fused_f.iou_counts)


@pytest.mark.parametrize("dtype", DTYPES)
def test_compat_modules_upcast_half_inputs(dev, dtype):
    """PixelwiseKLD and UncertaintyWeightedSegmentationLoss on fp16 / bf16 inputs: the values of their fp32 forms on x.float(),
    bit for bit, and the fp32 gradients cast to the input dtype, bit for bit."""
    from mspl_b200.loss_fns.segmentation_loss import PixelwiseKLD, UncertaintyWeightedSegmentationLoss
    n, k, h, w = 2, 5, 24, 40
    main, aux = _logits(n, k, h, w, dtype, dev, seed=71)
    tgt = _targets(n, k, h, w, False, dev, seed=72, invalid=False)
    up = torch.rand((n, h, w), generator=torch.Generator().manual_seed(73)).to(dev)
    m, a = main.clone().requires_grad_(True), aux.clone().requires_grad_(True)
    m32, a32 = main.float().requires_grad_(True), aux.float().requires_grad_(True)
    d, d32 = PixelwiseKLD()(m, a), PixelwiseKLD()(m32, a32)
    assert d.dtype == torch.float32 and torch.equal(d, d32)
    d.backward(up)
    d32.backward(up)
    assert torch.equal(m.grad, m32.grad.to(dtype)) and torch.equal(a.grad, a32.grad.to(dtype))

    crit = UncertaintyWeightedSegmentationLoss(k, _cw(k, dev).clone())
    p, p32 = main.clone().requires_grad_(True), main.float().requires_grad_(True)
    u = up.to(dtype).requires_grad_(True)
    u32 = u.detach().float().requires_grad_(True)
    l, l32 = crit(p, tgt, u), crit(p32, tgt, u32)
    assert torch.equal(l, l32)
    (l * 3).backward()
    (l32 * 3).backward()
    assert torch.equal(p.grad, p32.grad.to(dtype)) and torch.equal(u.grad, u32.grad.to(dtype))


def test_half_rejections(ops, dev):
    """Mixed logit dtypes and fp64 are refused, as are more than eight classes in half precision; the fused-upsample loss
    still takes fp32 only."""
    from mspl_b200.loss_fns.segmentation_loss import FusedUpsampleUncertaintyWeightedLoss
    n, k, h, w = 1, 5, 8, 16
    main, aux = _logits(n, k, h, w, torch.bfloat16, dev, seed=81)
    tgt = _targets(n, k, h, w, False, dev, seed=82)
    cw = _cw(k, dev)
    with pytest.raises(ValueError):
        ops.uw_ce_fwd_bwd(main, aux.half(), tgt, cw)
    with pytest.raises(ValueError):
        ops.uw_ce_loss(main.half(), aux, tgt, cw)
    with pytest.raises(ValueError):
        ops.uw_ce_fwd_bwd(main.double(), aux.double(), tgt, cw)
    with pytest.raises(ValueError):
        ops.uw_ce_fwd_bwd(main.float(), aux.float(), tgt, cw, grad_scale_dev=torch.ones(1, device=dev))
    m9, a9 = _logits(n, 9, h, w, torch.float16, dev, seed=83)
    with pytest.raises(NotImplementedError):
        ops.uw_ce_fwd_bwd(m9, a9, tgt, torch.ones(9, device=dev))
    lowres = FusedUpsampleUncertaintyWeightedLoss(k, cw.clone())
    with pytest.raises(ValueError):
        lowres(main[:, :, ::2, ::2].contiguous(), aux[:, :, ::2, ::2].contiguous(), tgt)
