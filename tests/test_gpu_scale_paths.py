"""-m gpu: the kernel paths the small oracle cases never reach, against the same CPU / fp64 oracles and tolerances as
tests/test_gpu_parity.py -- persistent CTAs that run more than one tile or grid-stride pass, the 8-target-class (KT = 8)
instantiations of K1, K4-lowres with 4-, 2- and 1-row tiles, NIDLoss at its bin limits, the run-time-C loss kernels behind
the K > 8 training route, and per-source tensors of more than 2^31 elements.

Every case runs its call under torch.profiler and asserts from the recorded launches that the targeted instantiation ran and
that its loop repeats (more tiles or pixel groups than the launched grid covers in one pass), so a dispatch change or an
alignment fallback cannot turn a case into a copy of a small one."""
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

SOURCES = (("camvid", 13), ("cityscapes", 20), ("forest", 5))


def _per_image(fn, n, *args):
    """A mean-over-pixels loss evaluated image by image (bounded host memory): every image has the same pixel count, so the
    global loss is the mean of the per-image losses and each image's gradient is its own divided by n (the global divisor)."""
    loss, gm, ga = 0.0, [], []
    for i in range(n):
        l, g1, g2 = fn(*[a[i:i + 1] for a in args[:-1]], args[-1], dtype=torch.float64)
        loss += float(l) / n
        gm.append(g1 / n)
        ga.append(g2 / n)
    return loss, torch.cat(gm), torch.cat(ga)


# ---- K4-lowres -----------------------------------------------------------------------------------------------------------
def _lowres_smem(K, TR, hm, wm, ha, wa, H, W):
    """lowres_smem_bytes (uw_loss_lowres.cuh) of the forward+backward kernel for a TR-row tile, in the kernel's fp32 arithmetic."""
    f = np.float32
    rhm, rha = (f(hm - 1) / f(H - 1), f(ha - 1) / f(H - 1)) if H > 1 else (f(0), f(0))
    nrm, nra = min(hm, int(rhm * f(TR - 1)) + 3), min(ha, int(rha * f(TR - 1)) + 3)
    src, tn = K * (nrm * wm + nra * wa), K * TR * max(wm, wa)
    tables = 4 * W + (wm + 1) + (wa + 1) + 4 * TR + K + 4 * W + (nrm + nra) * TR
    return 4 * (2 * K * TR * W + max(src, tn) + tables)


def _lowres_tr(dev, K, hm, wm, ha, wa, H, W):
    """The tile height launch_uw_ce_lowres picks: the tallest of 8, 4, 2, 1 whose shared memory fits one CTA."""
    limit = torch.cuda.get_device_properties(dev).shared_memory_per_block_optin
    return next(tr for tr in (8, 4, 2, 1) if _lowres_smem(K, tr, hm, wm, ha, wa, H, W) <= limit)


def _lowres_inputs(b, k, hm, wm, ha, wa, h, w, seed):
    gen = torch.Generator().manual_seed(seed)
    main_lr = 3.0 * torch.randn(b, k, hm, wm, generator=gen)
    aux_lr = 3.0 * torch.randn(b, k, ha, wa, generator=gen)
    target = torch.randint(0, k, (b, h, w), generator=gen)
    cw = torch.rand(k, generator=gen) * 3
    cw[k - 1] = 0.0
    return main_lr, aux_lr, target, cw


def _check_lowres(out3, dm, da, ref):
    l64, gm64, ga64 = ref
    assert abs(out3[0].item() - l64) <= RTOL * abs(l64)
    assert abs(out3[0].item() - (20 * out3[1].item() + out3[2].item())) <= 1e-5 * abs(l64)
    scale = float(max(gm64.abs().max(), ga64.abs().max()))          # tolerances of test_fused_upsample_loss_matches_oracle
    torch.testing.assert_close(dm.cpu().double(), gm64, rtol=1e-4, atol=5e-5 * scale)
    torch.testing.assert_close(da.cpu().double(), ga64, rtol=1e-4, atol=5e-5 * scale)
    return scale


@pytest.mark.parametrize("k,tr", [(5, 8), (8, 4)])
def test_lowres_loss_training_batch(ops, dev, sms, launches, k, tr):
    """ESPDNetUE geometry (256x480 from 128x240 / 64x120) at 24 images: 768 tiles, about five per CTA with the backward and
    more than one per CTA forward-only.  Against the fp64 oracle; int64 and uint8 targets; run-to-run; forward-only.  With
    K = 8 the gradient tile leaves room for 4-row tiles only, where an aux row can collect three shares: equal to rounding."""
    b, h, w, (hm, wm), (ha, wa) = 24, 256, 480, (128, 240), (64, 120)
    assert _lowres_tr(dev, k, hm, wm, ha, wa, h, w) == tr
    n_tiles = b * -(-h // tr)
    assert n_tiles >= 3 * sms
    main_lr, aux_lr, target, cw = _lowres_inputs(b, k, hm, wm, ha, wa, h, w, seed=k)
    ref = _per_image(O.training_loss_lowres_and_grads, b, main_lr, aux_lr, target, cw)
    m, a, t64, c = main_lr.to(dev), aux_lr.to(dev), target.to(dev), cw.to(dev)
    (out3, dm, da), ks = launches(lambda: ops.uw_ce_lowres_fwd_bwd(m, a, t64, c))
    kern = _the(ks, "uw_ce_lowres_kernel<%d,true,long>" % k)
    assert 0 <= kern.smem - _lowres_smem(k, tr, hm, wm, ha, wa, h, w) < 2048          # the TR-row carve-up was launched
    _repeats(kern, n_tiles)
    scale = _check_lowres(out3, dm, da, ref)
    (out8, dm8, da8), ks = launches(lambda: ops.uw_ce_lowres_fwd_bwd(m, a, t64.to(torch.uint8), c))
    _repeats(_the(ks, "uw_ce_lowres_kernel<%d,true,unsignedchar>" % k), n_tiles)
    out3b, dmb, dab = ops.uw_ce_lowres_fwd_bwd(m, a, t64, c)
    assert torch.equal(out8, out3) and torch.equal(out3b, out3)    # per-CTA sums reduced in a fixed order
    if tr == 8:
        # at most two shares per low-resolution element, and two adds onto zero commute: bit for bit (DESIGN section 4)
        for x, y in ((dm8, dm), (da8, da), (dmb, dm), (dab, da)):
            assert torch.equal(x, y)
    else:
        for x, y in ((dm8, dm), (da8, da), (dmb, dm), (dab, da)):
            torch.testing.assert_close(x, y, rtol=1e-5, atol=1e-6 * scale)
    (outf, none_m, none_a), ks = launches(lambda: ops.uw_ce_lowres_fwd_bwd(m, a, t64, c, backward=False))
    _repeats(_the(ks, "uw_ce_lowres_kernel<%d,false,long>" % k), n_tiles)
    assert none_m is None and none_a is None
    # the forward-only grid is wider (no gradient tile): the same per-tile terms summed over a different CTA partition
    torch.testing.assert_close(outf, out3, rtol=1e-6, atol=0)


@pytest.mark.parametrize("tr,b,w", [(4, 16, 768), (2, 8, 1024), (1, 4, 1536)])
def test_lowres_loss_short_tiles(ops, dev, sms, launches, tr, b, w):
    """Images too wide for 8-row gradient tiles (x2 / x4 heads, K = 5): 4-, 2- and 1-row tiles, where a low-resolution row
    collects shares from three or more tiles; 512 tiles each.  Against the fp64 oracle, run-to-run equal to rounding."""
    k, h = 5, 128
    hm, wm, ha, wa = h // 2, w // 2, h // 4, w // 4
    assert _lowres_tr(dev, k, hm, wm, ha, wa, h, w) == tr
    n_tiles = b * -(-h // tr)
    assert n_tiles >= 3 * sms
    main_lr, aux_lr, target, cw = _lowres_inputs(b, k, hm, wm, ha, wa, h, w, seed=10 + tr)
    ref = _per_image(O.training_loss_lowres_and_grads, b, main_lr, aux_lr, target, cw)
    m, a, t, c = main_lr.to(dev), aux_lr.to(dev), target.to(dev), cw.to(dev)
    (out3, dm, da), ks = launches(lambda: ops.uw_ce_lowres_fwd_bwd(m, a, t, c))
    kern = _the(ks, "uw_ce_lowres_kernel<5,true,long>")
    assert 0 <= kern.smem - _lowres_smem(k, tr, hm, wm, ha, wa, h, w) < 2048
    _repeats(kern, n_tiles)
    scale = _check_lowres(out3, dm, da, ref)
    out3b, dmb, dab = ops.uw_ce_lowres_fwd_bwd(m, a, t, c)
    assert torch.equal(out3b, out3)
    torch.testing.assert_close(dmb, dm, rtol=1e-5, atol=1e-6 * scale)
    torch.testing.assert_close(dab, da, rtol=1e-5, atol=1e-6 * scale)


# ---- NIDLoss ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("image_bins,label_bins,channels", [(16, 5, 5), (32, 8, 10)])
def test_nid_loss_beyond_one_grid_pass(dev, launches, image_bins, label_bins, channels):
    """B = 2 at 512x1024: 524,288 positions, two passes of the 1,024-CTA forward grid and of the backward grid.  The bin
    limits (32 / 8) with more label logits than label bins.  fp64 oracle + autograd, tolerances of
    test_nid_loss_full_size_vs_oracle; a wide label window (0.05) keeps the gradient dense."""
    from mspl_b200.loss_fns.segmentation_loss import NIDLoss
    b, h, w = 2, 512, 1024
    gen = torch.Generator().manual_seed(image_bins + channels)
    camera = torch.rand(b, 3, h, w, generator=gen)
    label = 0.004 * torch.randn(b, channels, h, w, generator=gen)
    lab64 = label.double().requires_grad_(True)
    want = O.nid_loss(camera.double(), lab64, image_bins, label_bins, 0.005, 0.05)
    gw, = torch.autograd.grad(want, lab64)
    ld = label.to(dev).requires_grad_(True)
    crit = NIDLoss(image_bins, label_bins, 0.005, 0.05)

    def step():
        loss = crit(camera.to(dev), ld)
        loss.backward()
        return loss
    got, ks = launches(step)
    _repeats(_the(ks, "nid_forward_kernel"), h * w, 256)
    _repeats(_the(ks, "nid_backward_kernel"), h * w, 256)
    assert abs(got.item() - want.item()) <= 1e-4
    torch.testing.assert_close(ld.grad.cpu().double(), gw, rtol=1e-3, atol=1e-4 * float(gw.abs().max()))


# ---- K1 with 6-8 target classes ------------------------------------------------------------------------------------------
def _sources(n, h, w, seed, num_classes):
    """Three sources (13 / 20 / 5 classes); K = 5 uses the greenhouse tables, other K random tables onto [0, K)."""
    gen = torch.Generator().manual_seed(seed)
    mains, auxs, luts = [], [], []
    for i, (nm, c) in enumerate(SOURCES):
        m, a = O.synthetic_logits(n, c, h, w, seed=seed + i)
        mains.append(m), auxs.append(a)
        luts.append(O.LUTS[nm] if num_classes == 5 else torch.randint(0, num_classes, (c,), generator=gen).numpy())
    return mains, auxs, luts


@pytest.mark.parametrize("policy", ["all", "half", "prob", 2])
def test_k1_eight_classes_full_size_batch(ops, dev, sms, launches, policy):
    """The KT = 8 counterpart of test_full_size_batch_against_the_oracle: 8 x 256x480, three sources on random tables onto
    K = 8 with ignore class 6 -- the 3-stage ring and the 8-class tally over 1,024 tiles (about seven per CTA).  Plus the
    labels-only kernel, and the scalar fallback (4-byte-offset views) bit for bit against the TMA kernel."""
    n, h, w, K, ignore = 8, 256, 480, 8, 6
    n_tiles = n * -(-(h * w) // 960)
    assert n_tiles >= 3 * sms
    mains, auxs, luts = _sources(n, h, w, 700, K)
    with _oracle_settings(ignore):
        ref = O.fuse_sources(mains, auxs, luts, policy, K, ignore)
    md, ad = [m.to(dev) for m in mains], [a.to(dev) for a in auxs]
    r, ks = launches(lambda: ops.fuse_sources(md, ad, luts, policy=policy, num_classes=K, ignore_label=ignore))
    _repeats(_the(ks, "fuse_sources_tma_kernel<15,2,5,3,8,"), n_tiles)
    _check_fusion(ops, r, ref, K, ignore)
    if policy != "prob":
        kw = dict(want_conf=False, want_unc=False, want_conf_hist=False, count_marginal=False)
        lean, ks = launches(lambda: ops.fuse_sources(md, ad, luts, policy=policy, num_classes=K, ignore_label=ignore, **kw))
        _repeats(_the(ks, "fuse_labels_tma_kernel<15,2,5,3,8>"), n_tiles)
        assert not bool(((lean.label.cpu() != ref["label"]) & ~ref["marginal"]).any())
        assert torch.equal(lean.label, r.label) and torch.equal(lean.class_hist, r.class_hist)
    offs = []
    for t in md + ad:
        buf = torch.empty(t.numel() + 1, device=dev)
        buf[1:] = t.reshape(-1)
        offs.append(buf[1:].view(t.shape))                                 # 4-byte aligned only
    s, ks = launches(lambda: ops.fuse_sources(offs[:3], offs[3:], luts, policy=policy, num_classes=K, ignore_label=ignore))
    _repeats(_the(ks, "fuse_sources_direct_kernel<5,8,"), n * h * w, 256)
    assert torch.equal(s.label, r.label) and torch.equal(s.conf, r.conf) and torch.equal(s.unc, r.unc)
    assert torch.equal(s.class_hist, r.class_hist) and torch.equal(s.conf_hist, r.conf_hist)
    assert int(s.marginal) == int(r.marginal)


@pytest.mark.parametrize("K", [5, 8])
def test_k1_partial_tiles_many_per_cta(ops, dev, sms, launches, K):
    """250x484 = 121,000 pixels: 126 whole 960-pixel tiles and a partial one per image, six images -- each CTA runs partial
    tiles followed by whole ones of the next image."""
    n, h, w = 6, 250, 484
    ignore = 4 if K == 5 else 6
    assert (h * w) % 960 != 0 and (h * w) % 4 == 0
    n_tiles = n * -(-(h * w) // 960)
    assert n_tiles >= 3 * sms
    mains, auxs, luts = _sources(n, h, w, 800 + K, K)
    md, ad = [m.to(dev) for m in mains], [a.to(dev) for a in auxs]
    for policy in ("half", "prob"):
        with _oracle_settings(ignore):
            ref = O.fuse_sources(mains, auxs, luts, policy, K, ignore)
        r, ks = launches(lambda: ops.fuse_sources(md, ad, luts, policy=policy, num_classes=K, ignore_label=ignore))
        _repeats(_the(ks, "fuse_sources_tma_kernel<15,2,5,%d,%d,true>" % (4 if K == 5 else 3, K)), n_tiles)
        _check_fusion(ops, r, ref, K, ignore)


# ---- K1-lowres -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,out_size,main_size,aux_size,policies,fragment", [
    (8, (256, 480), (128, 240), (64, 120), ("all", "prob"), "fuse_sources_lowres_kernel<15,2,5,4,8,"),
    # 3 rows x 256 main floats > the fixed 768-float class stride: the run-time-stride K <= 5 instantiation
    (5, (256, 512), (128, 256), (64, 128), ("half",), "fuse_sources_lowres_kernel<15,2,5,4,5,true,0,0>"),
])
def test_k1_lowres_at_scale(ops, dev, sms, launches, K, out_size, main_size, aux_size, policies, fragment):
    """8 images of a network's pre-upsample heads against upsample-then-fuse on the CPU, with the parity definition of
    test_fuse_sources_lowres (near-ties below 1e-5 excused, floats 1e-4 relative)."""
    n = 8
    ignore = 4 if K == 5 else 6
    n_tiles = n * -(-(out_size[0] * out_size[1]) // 960)
    assert n_tiles >= 3 * sms
    gen = torch.Generator().manual_seed(out_size[1] + K)
    mains, auxs, luts = [], [], []
    for nm, c in SOURCES:
        mains.append((3 * torch.randn(n, c, *main_size, generator=gen) + 3 * torch.randn(n, c, 1, 1, generator=gen)).contiguous())
        auxs.append(3 * torch.randn(n, c, *aux_size, generator=gen))
        luts.append(O.LUTS[nm] if K == 5 else torch.randint(0, K, (c,), generator=gen).numpy())
    md, ad = [m.to(dev) for m in mains], [a.to(dev) for a in auxs]
    for policy in policies:
        with _oracle_settings(ignore, margin=1e-5):
            ref = O.fuse_sources_lowres(mains, auxs, luts, out_size, policy, K, ignore)
        r, ks = launches(lambda: ops.fuse_sources_lowres(md, ad, luts, out_size, policy=policy, num_classes=K, ignore_label=ignore))
        _repeats(_the(ks, fragment), n_tiles)
        _check_fusion(ops, r, ref, K, ignore, conf_rtol=1e-4, conf_atol=1e-6, unc_rtol=1e-4, unc_atol=1e-5)


# ---- the K > 8 training route: PixelwiseKLD + UncertaintyWeightedSegmentationLoss -----------------------------------------
@pytest.mark.parametrize("shape", [(12, 256, 480), (4, 251, 483)], ids=["aligned", "unaligned"])
@pytest.mark.parametrize("C", [9, 13, 20])
def test_reference_modules_above_eight_classes(ops, dev, launches, C, shape):
    """The route ops.uw_ce_loss points K > 8 to: the run-time-C kernels (uw_loss_kernel, softmax_kld_kernel's KLD-only
    branch, kld_bwd_kernel) over more than one grid-stride pass, vectorised (P = 4) and, with H*W % 4 != 0, scalar.  The
    training expression against the fp64 oracle with the tolerances of test_reference_named_modules; K0 / get_output."""
    from mspl_b200 import uest_seg_multi_os as U
    from mspl_b200.loss_fns.segmentation_loss import PixelwiseKLD, UncertaintyWeightedSegmentationLoss
    n, h, w = shape
    P = 4 if (h * w) % 4 == 0 else 1
    groups = n * h * w // P
    main, aux = O.synthetic_logits(n, C, h, w, seed=900 + C)
    gen = torch.Generator().manual_seed(C)
    target = torch.randint(0, C, (n, h, w), generator=gen)
    cw = torch.rand(C, generator=gen) + 0.5
    crit = UncertaintyWeightedSegmentationLoss(C, class_weights=cw.to(dev), ignore_idx=C - 1, device=dev)
    l64, gm64, ga64 = _per_image(O.training_loss_and_grads, n, main, aux, target, crit.class_weights.cpu())
    pred, pred_aux, t = main.to(dev).requires_grad_(True), aux.to(dev).requires_grad_(True), target.to(dev)

    def step():
        kld = PixelwiseKLD()(pred, pred_aux)
        loss = crit(pred + 0.5 * pred_aux, t, kld) * 20 + kld.mean()
        loss.backward()
        return loss
    loss, ks = launches(step)
    for fragment in ("softmax_kld_kernel<%d>" % P, "uw_loss_kernel<%d,false>" % P, "uw_loss_kernel<%d,true>" % P,
                     "kld_bwd_kernel<%d>" % P):
        _repeats(_the(ks, fragment), groups, 256)
    assert abs(loss.item() - l64) <= RTOL * abs(l64)
    scale = float(gm64.abs().max())
    torch.testing.assert_close(pred.grad.cpu().double(), gm64, rtol=1e-4, atol=1e-5 * scale)
    torch.testing.assert_close(pred_aux.grad.cpu().double(), ga64, rtol=1e-4, atol=1e-5 * scale)
    # K0: softmax(main + 0.5 aux) and the KLD map, with and without the probability output, and get_output's image 0
    m, a = main.to(dev), aux.to(dev)
    prob_ref = torch.softmax(main.double() + 0.5 * aux.double(), dim=1)
    kld_ref = O.pixelwise_kld(main.double(), aux.double())
    (prob, kld), ks = launches(lambda: ops.softmax_kld(m, a))
    _repeats(_the(ks, "softmax_kld_kernel<%d>" % P), groups, 256)
    torch.testing.assert_close(prob.cpu().double(), prob_ref, rtol=RTOL, atol=1e-9)
    torch.testing.assert_close(kld.cpu().double(), kld_ref, rtol=RTOL, atol=KLD_ATOL)
    _, kld_only = ops.softmax_kld(m, a, want_prob=False)
    torch.testing.assert_close(kld_only.cpu().double(), kld_ref, rtol=RTOL, atol=KLD_ATOL)
    out, k0 = U.get_output(lambda x: (m, a), torch.zeros(1, 3, 4, 4), device=dev)
    np.testing.assert_allclose(out, prob_ref[0].numpy(), rtol=RTOL, atol=1e-9)
    np.testing.assert_allclose(k0, kld_ref[0].numpy(), rtol=RTOL, atol=KLD_ATOL)
    with pytest.raises(NotImplementedError):
        ops.uw_ce_loss(m, a, t, crit.class_weights)


# ---- per-source tensors over 2^31 elements -------------------------------------------------------------------------------
def _need_device_memory(dev, gib):
    if torch.cuda.get_device_properties(dev).total_memory < 80 * 2 ** 30:
        pytest.skip("needs ~%d GB of device memory" % gib)


def _fill_normal(shape, dev, gen, std=3.0, step=128):
    """A (N, ...) device tensor of N(0, std^2) values written in slices of images (no tensor-sized temporaries)."""
    x = torch.empty(shape, device=dev)
    for lo in range(0, shape[0], step):
        x[lo:lo + step].normal_(0.0, std, generator=gen)
    return x


def test_k1_source_over_2_31_elements(ops, dev, launches):
    """A 20-class source over 874 images of 480x256: each head is 2,147,942,400 floats, so the offsets of the last images
    exceed 2^31.  The first two and the last two images against the CPU oracle; class counts against the label map."""
    _need_device_memory(dev, 20)
    n, c, h, w = 874, 20, 256, 480
    assert n * c * h * w > 2 ** 31
    gen = torch.Generator(device=dev).manual_seed(2031)
    main = _fill_normal((n, c, h, w), dev, gen)
    aux = _fill_normal((n, c, h, w), dev, gen)
    lut = O.ID_CITYSCAPES_TO_GREENHOUSE
    r, ks = launches(lambda: ops.fuse_sources([main], [aux], [lut], policy="half"))
    _repeats(_the(ks, "fuse_sources_tma_kernel<15,2,5,4,5,"), n * -(-(h * w) // 960))
    assert torch.equal(r.class_hist, torch.bincount(r.label.reshape(-1).long(), minlength=5))
    for sl in (slice(0, 2), slice(n - 2, n)):
        ref = O.fuse_sources([main[sl].cpu()], [aux[sl].cpu()], [lut], "half")
        lab = r.label[sl].cpu()
        diff = lab != ref["label"]
        assert not bool((diff & ~ref["marginal"]).any())
        torch.testing.assert_close(r.conf[sl].cpu()[~diff], ref["conf"][~diff], rtol=RTOL, atol=1e-7)
        torch.testing.assert_close(r.unc[sl].cpu(), ref["unc"], rtol=RTOL, atol=KLD_ATOL)


def test_k4_tensor_over_2_31_elements(ops, dev, launches):
    """K = 8 over 2,185 images of 480x256: main, aux and both gradients hold 2,147,942,400 floats each.  The loss against an
    fp64 evaluation of the oracle's expression on the device (in slices), the first and the last image's gradients against
    the fp64 CPU oracle with the global pixel count as the divisor."""
    _need_device_memory(dev, 40)
    n, k, h, w = 2185, 8, 256, 480
    assert n * k * h * w > 2 ** 31
    gen = torch.Generator(device=dev).manual_seed(2032)
    main = _fill_normal((n, k, h, w), dev, gen)
    aux = _fill_normal((n, k, h, w), dev, gen)
    target = torch.randint(0, k, (n, h, w), device=dev, generator=gen, dtype=torch.uint8)
    cw = torch.linspace(0.5, 2.0, k, device=dev)
    (out3, dm, da), ks = launches(lambda: ops.uw_ce_fwd_bwd(main, aux, target, cw))
    _repeats(_the(ks, "uw_ce_fused_kernel<2,8,true,unsignedchar,false>"), n * h * w // 2, 256)
    total, step = 0.0, 64
    for lo in range(0, n, step):
        sl = slice(lo, min(n, lo + step))
        part = O.training_loss(main[sl].double(), aux[sl].double(), target[sl].long(), cw.double())
        total += float(part) * (sl.stop - sl.start) / n
    assert abs(out3[0].item() - total) <= RTOL * abs(total)
    for i in (0, n - 1):
        _, gm64, ga64 = O.training_loss_and_grads(main[i:i + 1].cpu(), aux[i:i + 1].cpu(), target[i:i + 1].cpu().long(), cw.cpu(),
                                                  dtype=torch.float64)
        gm64, ga64 = gm64 / n, ga64 / n
        scale = float(gm64.abs().max())
        torch.testing.assert_close(dm[i:i + 1].cpu().double(), gm64, rtol=2e-5, atol=2e-6 * scale)
        torch.testing.assert_close(da[i:i + 1].cpu().double(), ga64, rtol=2e-5, atol=2e-6 * scale)
