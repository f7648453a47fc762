"""TEST INFRASTRUCTURE ONLY -- writes tests/golden/*.npz from the LIVE reference.

Run in the build container (the only place /root/reference exists):

    PYTHONDONTWRITEBYTECODE=1 python -m oracle.make_golden

Every output array in the fixtures is produced by calling the reference's own functions unmodified
(uest_seg_multi_os.get_output / merge_outputs / transfer_output_to_greenhouse, the greenhouse LUTs,
loss_fns.segmentation_loss.PixelwiseKLD / UncertaintyWeightedSegmentationLoss and autograd).  The
inputs are stored beside them so that nothing has to be regenerated on the GPU box.
"""
import os
import sys

import numpy as np
import torch

from oracle.ref_import import FixedLogitsModel, build_espdnetue, load_reference

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
SOURCES = (("camvid", 13), ("cityscapes", 20), ("forest", 5))
POLICIES = ("half", "all", 1, 2, 3)


def _ref_label_gen(ref, mains, auxs, names, policy):
    """The reference's per-image loop body (uest_seg_multi_os.py:897-921) called through its own functions."""
    U = ref.uest
    luts = {"camvid": ref.greenhouse.id_camvid_to_greenhouse,
            "cityscapes": ref.greenhouse.id_cityscapes_to_greenhouse,
            "forest": ref.greenhouse.id_forest_to_greenhouse}
    n = mains[0].shape[0]
    labels, class_array = [], np.zeros(5)
    for i in range(n):
        per_source = []
        for m, a, name in zip(mains, auxs, names):
            output, _ = U.get_output(FixedLogitsModel(m[i:i + 1], a[i:i + 1]), torch.zeros(1), device='cpu')
            output = output.transpose(1, 2, 0)
            amax = np.asarray(np.argmax(output, axis=2), dtype=np.uint8)
            per_source.append(luts[name][amax])
        lab = U.merge_outputs(np.array(per_source), seg_classes=5, thresh=policy)
        for k in range(5):
            class_array[k] += (lab == k).sum()
        labels.append(lab.astype(np.uint8))
    return np.stack(labels), class_array


def _logits(n, c, h, w, gen, sigma=3.0, corr=True):
    main = sigma * torch.randn(n, c, h, w, generator=gen) + sigma * torch.randn(n, c, 1, 1, generator=gen)
    if corr:
        aux = main + 0.5 * sigma * torch.randn(n, c, h, w, generator=gen)
    else:
        aux = sigma * torch.randn(n, c, h, w, generator=gen)
    return main.contiguous(), aux.contiguous()


def golden_multi_source(ref):
    """3-source (camvid 13 / cityscapes 20 / forest 5) label generation, all vote policies."""
    gen = torch.Generator().manual_seed(3)          # the reference's RANDSEED (uest_seg_multi_os.py:79)
    n, h, w = 2, 24, 40
    out = {}
    mains, auxs = [], []
    for name, c in SOURCES:
        m, a = _logits(n, c, h, w, gen)
        mains.append(m), auxs.append(a)
        out["main_" + name], out["aux_" + name] = m.numpy(), a.numpy()
    U = ref.uest
    for (name, c), m, a in zip(SOURCES, mains, auxs):
        sm, kl = [], []
        for i in range(n):
            o, k = U.get_output(FixedLogitsModel(m[i:i + 1], a[i:i + 1]), torch.zeros(1), device='cpu')
            sm.append(o), kl.append(k)
        out["softmax_" + name], out["kld_" + name] = np.stack(sm), np.stack(kl)
        lut = getattr(ref.greenhouse, "id_%s_to_greenhouse" % name)
        out["lut_" + name] = np.asarray(lut)
        out["gh_prob_" + name] = np.stack([U.transfer_output_to_greenhouse(lut, s) for s in sm])
    names = [s[0] for s in SOURCES]
    for pol in POLICIES:
        lab, ca = _ref_label_gen(ref, mains, auxs, names, pol)
        out["label_%s" % pol], out["class_array_%s" % pol] = lab, ca
    # 1- and 2-source subsets (S=1 is the generate_pseudo_label special case, S=2 exercises 'half' == 'all')
    lab, ca = _ref_label_gen(ref, mains[:1], auxs[:1], names[:1], None)
    out["label_s1"], out["class_array_s1"] = lab, ca
    lab, ca = _ref_label_gen(ref, mains[:2], auxs[:2], names[:2], "half")
    out["label_s2_half"], out["class_array_s2_half"] = lab, ca
    np.savez_compressed(os.path.join(GOLDEN_DIR, "multi_source_3src.npz"), **out)


def golden_adversarial(ref):
    """Pure ties (all-equal logits), +-80 magnitude logits, near one-hot +-30 logits."""
    gen = torch.Generator().manual_seed(1882)       # eval_label.py:280-281
    n, h, w = 1, 8, 16
    out = {}
    names = [s[0] for s in SOURCES]
    for tag in ("ties", "big", "onehot"):
        mains, auxs = [], []
        for name, c in SOURCES:
            if tag == "ties":
                m = torch.zeros(n, c, h, w)
                a = torch.zeros(n, c, h, w)
                m[:, :, :, w // 2:] = torch.randint(0, 2, (n, c, h, w - w // 2), generator=gen).float()
            elif tag == "big":
                m = 80.0 * torch.sign(torch.randn(n, c, h, w, generator=gen))
                a = 80.0 * torch.sign(torch.randn(n, c, h, w, generator=gen))
            else:
                idx = torch.randint(0, c, (n, 1, h, w), generator=gen)
                m = torch.full((n, c, h, w), -30.0).scatter_(1, idx, 30.0)
                a = m + 0.1 * torch.randn(n, c, h, w, generator=gen)
            mains.append(m.contiguous()), auxs.append(a.contiguous())
            out["%s_main_%s" % (tag, name)], out["%s_aux_%s" % (tag, name)] = m.numpy(), a.numpy()
            o, k = ref.uest.get_output(FixedLogitsModel(m, a), torch.zeros(1), device='cpu')
            out["%s_softmax_%s" % (tag, name)], out["%s_kld_%s" % (tag, name)] = o[None], k[None]
        for pol in ("half", "all"):
            lab, ca = _ref_label_gen(ref, mains, auxs, names, pol)
            out["%s_label_%s" % (tag, pol)], out["%s_class_array_%s" % (tag, pol)] = lab, ca
    np.savez_compressed(os.path.join(GOLDEN_DIR, "adversarial.npz"), **out)


def golden_config1(ref):
    """BASELINE config 1: 8 synthetic 480x256 images through a random-init 20-class ESPDNetUE
    (torch.manual_seed(3)), reference CPU path.  The full-resolution logits are 157 MB, so the fixture
    keeps one 16x32 window per image, which holds the file under 1 MB (every op on the path is per-pixel, so cropping
    commutes with it)."""
    model = build_espdnetue(20, seed=3)
    gen = torch.Generator().manual_seed(3)
    lut = ref.greenhouse.id_cityscapes_to_greenhouse
    h0, w0, hh, ww = 104, 216, 16, 32
    mains, auxs, sms, klds, labs = [], [], [], [], []
    class_array = np.zeros(5)
    with torch.no_grad():
        for i in range(8):
            image = torch.randn(1, 3, 256, 480, generator=gen)
            main, aux = model(image)
            output, kld = ref.uest.get_output(FixedLogitsModel(main, aux), image, device='cpu')
            amax = np.asarray(np.argmax(output.transpose(1, 2, 0), axis=2), dtype=np.uint8)
            lab = ref.uest.merge_outputs(np.array([lut[amax]]), seg_classes=5, thresh=None)
            for k in range(5):
                class_array[k] += (lab == k).sum()
            sl = (slice(h0, h0 + hh), slice(w0, w0 + ww))
            mains.append(main[0][:, sl[0], sl[1]].numpy().copy())
            auxs.append(aux[0][:, sl[0], sl[1]].numpy().copy())
            sms.append(output[:, sl[0], sl[1]].copy()), klds.append(kld[sl].copy())
            labs.append(lab[sl].astype(np.uint8))
    np.savez_compressed(os.path.join(GOLDEN_DIR, "config1_espdnetue_crop.npz"),
                        main=np.stack(mains), aux=np.stack(auxs), softmax=np.stack(sms), kld=np.stack(klds),
                        label=np.stack(labs), full_class_array=class_array, lut=np.asarray(lut),
                        window=np.array([h0, w0, hh, ww]))


def golden_loss(ref):
    """PixelwiseKLD + UncertaintyWeightedSegmentationLoss*20 + kld.mean() forward and autograd backward
    (uest_seg_multi_os.py:1020-1023), plus the two modules on their own."""
    gen = torch.Generator().manual_seed(3)
    b, k, h, w = 2, 5, 16, 24
    main, aux = _logits(b, k, h, w, gen)
    target = torch.randint(0, k, (b, h, w), generator=gen)
    out = dict(main=main.numpy(), aux=aux.numpy(), target=target.numpy())
    L = ref.seg_loss
    for tag, cw in (("flat", torch.ones(k)), ("normal", torch.tensor([0.0, 3.1, 7.7, 2.2, 9.0]))):
        cw = cw.clone()
        crit = L.UncertaintyWeightedSegmentationLoss(k, class_weights=cw, ignore_idx=4, device='cpu')
        m = main.clone().requires_grad_(True)
        a = aux.clone().requires_grad_(True)
        kld = L.PixelwiseKLD()(m, a)
        loss = crit(m + 0.5 * a, target, kld) * 20 + kld.mean()
        gm, ga = torch.autograd.grad(loss, (m, a))
        out["cw_" + tag] = cw.numpy()          # after the ctor's in-place zeroing of [ignore_idx]
        out["loss_" + tag] = loss.detach().numpy()
        out["grad_main_" + tag], out["grad_aux_" + tag] = gm.numpy(), ga.numpy()
        # the two modules separately, with independent inputs (generic drop-in contract)
        p = main.clone().requires_grad_(True)
        u = (aux[:, 0].abs()).clone().requires_grad_(True)
        l2 = crit(p, target, u)
        gp, gu = torch.autograd.grad(l2, (p, u))
        out["uw_u_" + tag], out["uw_loss_" + tag] = u.detach().numpy(), l2.detach().numpy()
        out["uw_grad_pred_" + tag], out["uw_grad_u_" + tag] = gp.numpy(), gu.numpy()
    d1 = main.clone().requires_grad_(True)
    d2 = aux.clone().requires_grad_(True)
    kl = L.PixelwiseKLD()(d1, d2)
    up = torch.randn(b, h, w, generator=gen)
    g1, g2 = torch.autograd.grad(kl, (d1, d2), grad_outputs=up)
    out["kld"], out["kld_upstream"], out["kld_grad1"], out["kld_grad2"] = kl.detach().numpy(), up.numpy(), g1.numpy(), g2.numpy()
    torch.autograd.set_detect_anomaly(False)    # the reference's forward switches it on globally (:156)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "loss_k5.npz"), **out)


def golden_miou(ref):
    """MIOU.get_iou (utilities/metrics/segmentation_miou.py:13-44) on logits and on label maps, with 255-labelled and
    out-of-range pixels, for 5 and 21 classes."""
    from utilities.metrics.segmentation_miou import MIOU
    gen = torch.Generator().manual_seed(3)
    out = {}
    for nc in (5, 21):
        logits = torch.randn(3, nc, 20, 28, generator=gen)
        logits[:, :, :2] = 0.0                                   # exact ties -> first maximal index
        target = torch.randint(0, nc + 2, (3, 20, 28), generator=gen)
        target[target == nc + 1] = 255                           # "ignore" pixels of the reference loaders
        inter, union = MIOU(num_classes=nc).get_iou(logits.clone(), target.clone())
        out["logits_%d" % nc], out["target_%d" % nc] = logits.numpy(), target.numpy()
        out["inter_%d" % nc], out["union_%d" % nc] = inter, union
        pred = torch.randint(0, nc + 1, (3, 20, 28), generator=gen)
        inter, union = MIOU(num_classes=nc).get_iou(pred.clone(), target.clone())
        out["pred_%d" % nc], out["inter_lab_%d" % nc], out["union_lab_%d" % nc] = pred.numpy(), inter, union
    np.savez_compressed(os.path.join(GOLDEN_DIR, "miou.npz"), **out)


def golden_nid(ref):
    """NIDLoss forward + autograd backward (loss_fns/segmentation_loss.py:54-144).  The reference hard-codes .to('cuda');
    in this GPU-less container Tensor.to is wrapped for the duration of the calls so that 'cuda' means 'cpu'."""
    orig_to = torch.Tensor.to

    def to_cpu(self, *a, **k):
        a = tuple('cpu' if (isinstance(x, str) and x.startswith('cuda')) else x for x in a)
        return orig_to(self, *a, **k)
    torch.Tensor.to = to_cpu
    try:
        gen = torch.Generator().manual_seed(3)
        out = {}
        cases = {"hard": dict(scale=3.0, kw={}),                                      # soft-argmax saturated: gradient vanishes
                 "soft": dict(scale=0.004, kw=dict(bw_label=0.05)),                   # soft labels, wide label windows: dense gradient
                 "bins8": dict(scale=0.004, kw=dict(image_bin=8, label_bin=4, bw_camera=0.02, bw_label=0.1))}
        for tag, cfg in cases.items():
            b, c, h, w = 3, 5, 12, 20
            camera = torch.rand(b, 3, h, w, generator=gen) * 1.2 - 0.1                    # some intensities outside [0,1]
            label = cfg["scale"] * torch.randn(b, c, h, w, generator=gen)
            kw = dict(image_bin=16, label_bin=5)
            kw.update(cfg["kw"])
            crit = ref.seg_loss.NIDLoss(**kw)
            lab = label.clone().requires_grad_(True)
            loss = crit(camera, lab)
            grad, = torch.autograd.grad(loss, lab)
            out["camera_" + tag], out["label_" + tag] = camera.numpy(), label.numpy()
            out["loss_" + tag], out["grad_" + tag] = loss.detach().numpy(), grad.numpy()
            out["cfg_" + tag] = np.array([kw["image_bin"], kw["label_bin"], kw.get("bw_camera", 0.005), kw.get("bw_label", 0.001)])
        np.savez_compressed(os.path.join(GOLDEN_DIR, "nid.npz"), **out)
    finally:
        torch.Tensor.to = orig_to


GREENHOUSE_ENCODING = (('end_of_plant', (0, 255, 0)), ('other_part_of_plant', (0, 255, 255)), ('artificial_objects', (255, 0, 0)),
                       ('ground', (255, 255, 0)), ('background', (0, 0, 0)))


class CapturingWriter:
    """Stands in for the TensorBoard SummaryWriter the reference writes its grids to."""

    def __init__(self):
        self.images = {}
        self.order = []

    def add_image(self, tag, img, epoch):
        self.images[tag] = np.asarray(img)
        self.order.append(tag)


def golden_visualization(ref):
    """in_training_visualization_img (utilities/utils.py:76-133) run live with a capturing writer: tuple predictions (KLD heat
    map + argmax of main + 0.5*aux) and plain-tensor predictions, greenhouse colour encoding."""
    from collections import OrderedDict
    gen = torch.Generator().manual_seed(3)
    enc = OrderedDict(GREENHOUSE_ENCODING)
    b, c, h, w = 3, 5, 20, 28
    images = torch.rand(b, 3, h, w, generator=gen)
    main = 3.0 * torch.randn(b, c, h, w, generator=gen)
    aux = main + 1.5 * torch.randn(b, c, h, w, generator=gen)
    labels = torch.randint(0, c, (b, h, w), generator=gen)
    out = dict(images=images.numpy(), main=main.numpy(), aux=aux.numpy(), labels=labels.numpy())
    wr = CapturingWriter()
    ref.utils.in_training_visualization_img(None, images.clone(), labels=labels.clone(), predictions=(main.clone(), aux.clone()),
                                            class_encoding=enc, writer=wr, epoch=0, data='train')
    for tag, img in wr.images.items():
        out["tuple_" + tag.replace('/', '_')] = img
    out["tuple_order"] = np.array(wr.order)
    wr = CapturingWriter()
    ref.utils.in_training_visualization_img(None, images.clone(), labels=None, predictions=main.clone(), class_encoding=enc, writer=wr,
                                            epoch=0, data='val')
    for tag, img in wr.images.items():
        out["tensor_" + tag.replace('/', '_')] = img
    out["tensor_order"] = np.array(wr.order)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "visualization.npz"), **out)


def golden_train_step(ref):
    """The per-iteration statements of train() that sit on the path, run by the LIVE reference for three batches
    (uest_seg_multi_os.py:1020-1049): kld = kld_layer(pred, pred_aux); loss = criterion(pred + 0.5*pred_aux, labels, kld) * 20
    + kld.mean(); inter, union = miou_class.get_iou(pred, labels); the two AverageMeters; iou = inter_meter.sum /
    (union_meter.sum + 1e-10); miou = iou[[1, 2, 3]].mean() * 100.  Fixture of FusedUncertaintyWeightedLoss(track_iou=True)."""
    from loss_fns.segmentation_loss import PixelwiseKLD, UncertaintyWeightedSegmentationLoss
    from utilities.metrics.segmentation_miou import MIOU
    from utilities.utils import AverageMeter
    gen = torch.Generator().manual_seed(17)
    k, b, h, w = 5, 2, 24, 40
    cw = torch.tensor([1.0, 2.0, 0.5, 1.5, 3.0])
    crit = UncertaintyWeightedSegmentationLoss(k, class_weights=cw.clone(), ignore_idx=4, device='cpu')
    kld_layer, miou_class = PixelwiseKLD(), MIOU(num_classes=k)
    inter_meter, union_meter = AverageMeter(), AverageMeter()
    out = {"class_weights": cw.numpy()}
    for i in range(3):
        pred, pred_aux = _logits(b, k, h, w, gen)
        labels = torch.randint(0, k, (b, h, w), generator=gen)
        if i == 1:
            labels[0, 0, :4] = 255                                        # one batch with pixels the metric drops
        loss_labels = labels.clone()
        loss_labels[loss_labels == 255] = 4                               # the loss needs in-range targets (torch.gather)
        p, q = pred.clone().requires_grad_(True), pred_aux.clone().requires_grad_(True)
        kld = kld_layer(p, q)
        loss = crit(p + 0.5 * q, loss_labels, kld) * 20 + kld.mean()
        loss.backward()
        inter, union = miou_class.get_iou(pred, labels)
        inter_meter.update(inter)
        union_meter.update(union)
        out.update({"main_%d" % i: pred.numpy(), "aux_%d" % i: pred_aux.numpy(), "labels_%d" % i: labels.numpy(),
                    "loss_labels_%d" % i: loss_labels.numpy(), "loss_%d" % i: np.float32(loss.item()),
                    "grad_main_%d" % i: p.grad.numpy(), "grad_aux_%d" % i: q.grad.numpy(), "inter_%d" % i: inter, "union_%d" % i: union})
    iou = inter_meter.sum / (union_meter.sum + 1e-10)
    out["iou"], out["miou"] = iou, np.float32(iou[[1, 2, 3]].mean() * 100)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "train_step.npz"), **out)


def main():
    ref = load_reference()
    if ref is None:
        sys.exit("reference tree not found; golden fixtures can only be generated in the build container")
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(1)
    only = sys.argv[1:]
    for fn in (golden_multi_source, golden_adversarial, golden_loss, golden_config1, golden_miou, golden_nid, golden_visualization, golden_train_step):
        if not only or fn.__name__.replace("golden_", "") in only:
            fn(ref)
    for f in sorted(os.listdir(GOLDEN_DIR)):
        print(f, os.path.getsize(os.path.join(GOLDEN_DIR, f)))


if __name__ == "__main__":
    main()
