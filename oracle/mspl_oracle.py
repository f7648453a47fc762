"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the MSPL pseudo-label / uncertainty-loss hot path.

This file is the checker, never the product: only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it.  ``mspl_b200`` must never
import it (tests/test_no_oracle_in_product.py enforces that).

It restates, op for op and in the reference's own arithmetic (PyTorch CPU fp32 + NumPy), the
reference functions on the path (paths relative to the reference tree):

  * ``get_output``                      uest_seg_multi_os.py:669-693
  * ``PixelwiseKLD.forward``            loss_fns/segmentation_loss.py:181-189
  * per-source argmax + LUT             uest_seg_multi_os.py:903-912, data_loader/segmentation/greenhouse.py:15-58
  * ``merge_outputs``                   uest_seg_multi_os.py:695-718
  * class histogram + class weights     uest_seg_multi_os.py:919-921, 942-950
  * ``transfer_output_to_greenhouse``   uest_seg_multi_os.py:1334-1350
  * ``UncertaintyWeightedSegmentationLoss`` loss_fns/segmentation_loss.py:146-175
  * the training-loss combination       uest_seg_multi_os.py:1020-1023
  * ``MIOU.get_iou``                    utilities/metrics/segmentation_miou.py:13-44
  * ``NIDLoss`` / ``SoftArgMax``        loss_fns/segmentation_loss.py:54-144

Parity status.  The functions above are PINNED: tests/test_oracle_vs_reference.py runs them against
the live reference in the build container, and tests/golden/*.npz hold outputs generated from the
live reference by oracle/make_golden.py.  The two [NEW] stages that have NO reference implementation
(probability fusion / confidence ``fuse_sources`` and class-balanced thresholds ``cb_thresholds`` /
``apply_thresholds``; SURVEY.md section 8 A4', A4'') are "parity unpinned": this file is their
definition.
"""
import numpy as np
import torch
import torch.nn.functional as F

# Source -> greenhouse class tables (values of data_loader/segmentation/greenhouse.py:15-58).
ID_CAMVID_TO_GREENHOUSE = np.array([4, 2, 2, 3, 3, 1, 2, 2, 2, 4, 4, 2, 4])
ID_CITYSCAPES_TO_GREENHOUSE = np.array([3, 3, 2, 2, 2, 2, 2, 2, 1, 3, 4, 4, 4, 2, 2, 2, 2, 2, 2, 4])
ID_FOREST_TO_GREENHOUSE = np.array([3, 1, 1, 2, 2])
LUTS = {"camvid": ID_CAMVID_TO_GREENHOUSE, "cityscapes": ID_CITYSCAPES_TO_GREENHOUSE,
        "forest": ID_FOREST_TO_GREENHOUSE}
NUM_GREENHOUSE_CLASSES = 5   # greenhouse.py:14
IGNORE_LABEL = 4             # uest_seg_multi_os.py:716

NEAR_TIE_MARGIN = 1e-6       # BASELINE.json north_star: top-2 probability margin below which a pixel is "marginal"


# --------------------------------------------------------------------------------------------
# Pinned restatements
# --------------------------------------------------------------------------------------------
def pixelwise_kld(dist1, dist2):
    """loss_fns/segmentation_loss.py:181-189 -- KL(softmax(dist1) || softmax(dist2)) per pixel."""
    p1 = F.softmax(dist1, dim=1)
    logp1 = F.log_softmax(dist1, dim=1)
    logp2 = F.log_softmax(dist2, dim=1)
    kld_i = p1 * logp1 - p1 * logp2
    return torch.sum(kld_i, dim=1)


def get_output_from_logits(pred, pred_aux):
    """uest_seg_multi_os.py:687-691 after the model call: returns (softmax(main+0.5*aux)[0] as
    ndarray (C,H,W) f32, kld[0] as ndarray (H,W) f32).  Batch element 0 only, like the reference."""
    output2 = pred + 0.5 * pred_aux
    output = F.softmax(output2, dim=-3).cpu().data[0].numpy()   # nn.Softmax2d == softmax over dim -3
    kld = pixelwise_kld(pred, pred_aux).cpu().data[0].numpy()
    return output, kld


def get_output(model, image, model_name='espdnetue', device='cpu'):
    """uest_seg_multi_os.py:669-693 (tuple or OrderedDict{'out','aux'} model outputs)."""
    out = model(image.to(device))
    if isinstance(out, dict):
        pred, pred_aux = out['out'], out['aux']
    else:
        pred, pred_aux = out[0], out[1]
    return get_output_from_logits(pred, pred_aux)


def argmax_to_greenhouse(output, lut):
    """uest_seg_multi_os.py:903-912: first-max argmax over classes of the (C,H,W) softmax map on a
    transposed view, cast to uint8, then the integer table lookup (-> int64 (H,W))."""
    out_t = output.transpose(1, 2, 0)
    amax = np.asarray(np.argmax(out_t, axis=2), dtype=np.uint8)
    return np.asarray(lut)[amax]


def vote_threshold(num_data, thresh=None):
    """uest_seg_multi_os.py:697-705: None/'half'/invalid -> S//2+1, 'all' -> S, int<=S -> itself.  The reference tests
    isinstance(thresh, int), which a bool passes: True counts as 1, False as 0 (no pixel becomes the ignore class)."""
    if thresh is None or thresh == 'half':
        return num_data // 2 + 1
    if thresh == 'all':
        return num_data
    if isinstance(thresh, int) and thresh <= num_data:
        return thresh
    return num_data // 2 + 1


def merge_outputs(amax_outputs, seg_classes=NUM_GREENHOUSE_CLASSES, thresh=None):
    """uest_seg_multi_os.py:695-718: per-pixel majority vote over (S,H,W) labels; pixels whose
    winning count is below the vote threshold become class 4."""
    amax_outputs = np.asarray(amax_outputs)
    t = vote_threshold(amax_outputs.shape[0], thresh)
    counts = np.array([(amax_outputs == k).sum(axis=0) for k in range(seg_classes)])
    lab = counts.argmax(axis=0)
    lab[counts.max(axis=0) < t] = IGNORE_LABEL
    return lab


def class_histogram(label, seg_classes=NUM_GREENHOUSE_CLASSES):
    """uest_seg_multi_os.py:919-921."""
    return np.array([(label == i).sum() for i in range(seg_classes)], dtype=np.float64)


def class_weights_from_histogram(class_array, weighting='normal'):
    """uest_seg_multi_os.py:942-950 -> float32 tensor."""
    class_array = np.array(class_array, dtype=np.float64)
    if weighting == 'normal':
        class_array = class_array / class_array.sum()
        w = 1 / (class_array + 1e-10)
        w[0] = 0.0
    else:
        w = np.ones(len(class_array))
    return torch.from_numpy(w).float()


def transfer_output_to_greenhouse(id_to_greenhouse, output_np, seg_classes=NUM_GREENHOUSE_CLASSES):
    """uest_seg_multi_os.py:1334-1350: G[0]=0, G[k]=max_{c:LUT[c]==k} P[c] (0 if none); float64 (K,H,W)."""
    id_to_greenhouse = np.asarray(id_to_greenhouse)
    shape = (1, output_np.shape[1], output_np.shape[2])
    out = np.zeros(shape)
    for k in range(1, seg_classes):
        sel = id_to_greenhouse == k
        plane = output_np[sel].max(axis=0).reshape(shape) if sel.sum() else np.zeros(shape)
        out = np.append(out, plane, axis=0)
    return out


def multi_source_labels(mains, auxs, luts, thresh=None, seg_classes=NUM_GREENHOUSE_CLASSES):
    """The per-image body of generate_pseudo_label_multi_model (uest_seg_multi_os.py:897-921) for a
    batch: mains/auxs are lists (one per source) of (N,C_s,H,W) f32 tensors.  Returns
    (labels (N,H,W) uint8, class_array float64 (K,))."""
    n_img = mains[0].shape[0]
    labels = []
    class_array = np.zeros(seg_classes)
    for i in range(n_img):
        per_source = []
        for m, a, lut in zip(mains, auxs, luts):
            output, _ = get_output_from_logits(m[i:i + 1], a[i:i + 1])
            per_source.append(argmax_to_greenhouse(output, lut))
        lab = merge_outputs(np.array(per_source), seg_classes, thresh)
        class_array += class_histogram(lab, seg_classes)
        labels.append(lab.astype(np.uint8))
    return np.stack(labels), class_array


def uw_segmentation_loss(pred, target, u_weight, class_weights):
    """UncertaintyWeightedSegmentationLoss.forward, loss_fns/segmentation_loss.py:155-175 (without the
    global anomaly-mode switch at :156): mean over ALL pixels of w[t] * (-log_softmax(pred)[t]) * exp(-u)."""
    b, _, h, w = pred.shape
    logp = -F.log_softmax(pred, dim=1)
    logp = logp * class_weights.reshape(1, -1, 1, 1).expand(b, -1, h, w)
    logp = logp.gather(1, target.view(b, 1, h, w))
    logp = logp * torch.exp(-u_weight.reshape(b, 1, h, w))
    return logp.mean()


def make_class_weights(num_classes, class_weights=None, ignore_idx=None):
    """UncertaintyWeightedSegmentationLoss.__init__, loss_fns/segmentation_loss.py:147-153: zeroes the
    ignore entry IN PLACE on the caller's tensor."""
    w = class_weights if class_weights is not None else torch.ones(num_classes)
    if ignore_idx is not None:
        w[ignore_idx] = 0.0
    return w


def training_loss(pred, pred_aux, labels, class_weights, alpha=20.0):
    """uest_seg_multi_os.py:1020-1023 with --use-uncertainty: kld un-detached, CE term scaled by 20."""
    kld = pixelwise_kld(pred, pred_aux)
    return uw_segmentation_loss(pred + 0.5 * pred_aux, labels, kld, class_weights) * alpha + kld.mean()


def training_loss_and_grads(main, aux, labels, class_weights, alpha=20.0, dtype=torch.float32):
    """Loss and d(loss)/d(main), d(loss)/d(aux) by autograd on the restated forward."""
    m = main.detach().to(dtype).clone().requires_grad_(True)
    a = aux.detach().to(dtype).clone().requires_grad_(True)
    loss = training_loss(m, a, labels, class_weights.to(dtype), alpha)
    gm, ga = torch.autograd.grad(loss, (m, a))
    return loss.detach(), gm, ga


def miou_get_iou(output, target, num_classes=21, epsilon=1e-6):
    """MIOU.get_iou, utilities/metrics/segmentation_miou.py:13-44 (CPU tensors): returns (area_inter, area_union) float32
    ndarrays of length num_classes."""
    if isinstance(output, tuple):
        output = output[0]
    if output.dim() == 4:
        _, pred = torch.max(output, 1)
    else:
        pred = output
    pred = pred.type(torch.ByteTensor)
    target = target.type(torch.ByteTensor)
    pred = pred + 1          # shift by 1 so that 255 is 0 (uint8 wrap-around)
    target = target + 1
    pred = pred * (target > 0)
    inter = pred * (pred == target)
    area_inter = torch.histc(inter.float(), bins=num_classes, min=1, max=num_classes)
    area_pred = torch.histc(pred.float(), bins=num_classes, min=1, max=num_classes)
    area_mask = torch.histc(target.float(), bins=num_classes, min=1, max=num_classes)
    area_union = area_pred + area_mask - area_inter + epsilon
    return area_inter.numpy(), area_union.numpy()


def soft_arg_max(A, beta=500, epsilon=1e-12):
    """SoftArgMax.soft_arg_max, loss_fns/segmentation_loss.py:124-141 (device-agnostic): sum_i i * softmax(beta*A)_i."""
    A_max = torch.max(A, dim=1, keepdim=True)[0]
    A_exp = torch.exp((A - A_max) * beta)
    A_softmax = A_exp / (torch.sum(A_exp, dim=1, keepdim=True) + epsilon)
    indices = torch.arange(start=0, end=A.size()[1]).float().reshape(1, A.size()[1], 1, 1).to(A.dtype)
    return F.conv2d(A_softmax, indices)


def nid_loss(camera, label, image_bin=16, label_bin=4, bw_camera=0.005, bw_label=0.001, eps=1e-7):
    """NIDLoss.forward, loss_fns/segmentation_loss.py:54-118, without its hard-coded .to('cuda') calls.
    camera (B,3,H,W), label (B,C,H,W) logits.  Note the reference's quirk, kept here: the per-bin window responses are
    summed over the BATCH first (P_c is K x num_pixel), so the joint histogram couples images at the same pixel position."""
    camera_gray = torch.sum(camera, 1) / 3
    label_amax = soft_arg_max(label)
    label_amax = label_amax.reshape(label_amax.size()[0], label_amax.size()[2], label_amax.size()[3])
    num_pixel = camera_gray.size()[1] * camera_gray.size()[2]
    batch_size = camera_gray.size()[0]
    camera_1d = camera_gray.reshape(batch_size, -1)
    label_1d = torch.reshape(label_amax, (batch_size, -1))
    P_c = torch.zeros(image_bin, num_pixel, dtype=camera.dtype)
    P_l = torch.zeros(label_bin, num_pixel, dtype=camera.dtype)
    L_c = 1 / image_bin
    L_l = 1
    for k in range(0, image_bin):
        mu_k = L_c * (k + 1 / 2)
        PI_c = torch.sigmoid((camera_1d - mu_k + L_c / 2) / bw_camera) - torch.sigmoid((camera_1d - mu_k - L_c / 2) / bw_camera)
        P_c[k] = torch.sum(PI_c, 0)
        if k < label_bin:
            PI_l = torch.sigmoid((label_1d - k + L_l / 2) / bw_label) - torch.sigmoid((label_1d - k - L_l / 2) / bw_label)
            P_l[k] = torch.sum(PI_l, 0)
    norm = num_pixel * batch_size
    p_cl, p_c, p_l = torch.mm(P_c, torch.t(P_l)) / norm, torch.sum(P_c, 1) / norm, torch.sum(P_l, 1) / norm
    p_cl = p_cl / p_cl.sum()
    p_c = (p_c / p_c.sum()).reshape(-1, 1)
    p_l = (p_l / p_l.sum()).reshape(-1, 1)
    I = torch.sum(p_cl * (torch.log(p_cl + eps) - torch.log(torch.mm(p_c, torch.t(p_l)) + eps)))
    H = -torch.sum(p_cl * torch.log(p_cl + eps))
    nid = 1 - I / H
    return (nid - 0.95) * 20


# --------------------------------------------------------------------------------------------
# [NEW] stages -- no reference implementation ("parity unpinned"): this is the definition
# --------------------------------------------------------------------------------------------
def fuse_sources(mains, auxs, luts, policy='half', seg_classes=NUM_GREENHOUSE_CLASSES,
                 ignore=IGNORE_LABEL):
    """Batched fusion of S sources (SURVEY.md section 8 A4').

    Per source s: z = main + 0.5*aux, P = softmax(z), lab_s = LUT_s[first-argmax P], D_s = KLD(main, aux),
    G_s = transfer_output_to_greenhouse(LUT_s, P) in fp32.  F = (sum_s G_s) / S, U = (sum_s D_s) / S
    (sums in source order, fp32).
      policy 'half' / 'all' / int : label = merge_outputs vote; conf = F[label] where label != ignore else 0
      policy 'prob'               : label = first-argmax_k F ;  conf = max_k F
    Returns dict(label u8 (N,H,W), conf f32, unc f32, kld list of (N,H,W) f32, class_hist int64 (K,),
    marginal bool (N,H,W)).  ``marginal`` flags pixels where a different-but-legitimate fp32 rounding
    may change the label: for some source the softmax margin between the best class of its winning target and the
    best class of any OTHER target is < 1e-6 (SURVEY.md 8 A4'), or (policy 'prob') the top-2 margin of F < 1e-6.
    """
    S = len(mains)
    K = seg_classes
    n, _, h, w = mains[0].shape
    labs, klds = [], []
    Fsum = torch.zeros(n, K, h, w, dtype=torch.float32)
    Usum = torch.zeros(n, h, w, dtype=torch.float32)
    marginal = torch.zeros(n, h, w, dtype=torch.bool)
    for m, a, lut in zip(mains, auxs, luts):
        lut_t = torch.as_tensor(np.asarray(lut), dtype=torch.int64)
        z = m + 0.5 * a
        P = F.softmax(z, dim=1)
        amax = torch.from_numpy(np.argmax(P.numpy(), axis=1))       # first max, like np.argmax at :904
        labs.append(lut_t[amax])
        D = pixelwise_kld(m, a)
        klds.append(D)
        Usum = Usum + D
        G = torch.zeros(n, K, h, w, dtype=torch.float32)
        for k in range(1, K):
            sel = lut_t == k
            if bool(sel.any()):
                G[:, k] = P[:, sel].max(dim=1).values
        Fsum = Fsum + G
        # near-tie report: the best class of the winning TARGET against the best class of any other target (a near-tie between
        # two source classes that map to the same target cannot change the label)
        present = [k for k in range(K) if bool((lut_t == k).any())]
        if len(present) > 1:
            Gp = torch.stack([P[:, lut_t == k].max(dim=1).values for k in present], dim=1)
            top2 = torch.topk(Gp, 2, dim=1).values
            marginal |= (top2[:, 0] - top2[:, 1]) < NEAR_TIE_MARGIN
    Fm = Fsum / S
    U = Usum / S
    if policy == 'prob':
        label = torch.from_numpy(np.argmax(Fm.numpy(), axis=1))
        conf = Fm.max(dim=1).values
        t2 = torch.topk(Fm, 2, dim=1).values
        marginal |= (t2[:, 0] - t2[:, 1]) < NEAR_TIE_MARGIN
    else:
        stack = torch.stack(labs).numpy()                             # (S,N,H,W)
        label = torch.from_numpy(np.stack([merge_outputs(stack[:, i], K, policy) for i in range(n)]))
        conf = torch.gather(Fm, 1, label.unsqueeze(1)).squeeze(1)
        conf = torch.where(label == ignore, torch.zeros_like(conf), conf)
    class_hist = torch.bincount(label.reshape(-1), minlength=K)[:K]
    return dict(label=label.to(torch.uint8), conf=conf, unc=U, kld=klds, class_hist=class_hist,
                marginal=marginal, fused=Fm)


def upsample_heads(main_lr, aux_lr, out_size):
    """The closing statement of ESPDNetwithUncertaintyEstimation.forward, model/segmentation/espdnet_ue.py:301-302."""
    return (F.interpolate(main_lr, size=out_size, mode='bilinear', align_corners=True),
            F.interpolate(aux_lr, size=out_size, mode='bilinear', align_corners=True))


def fuse_sources_lowres(mains_lr, auxs_lr, luts, out_size, policy='half', seg_classes=NUM_GREENHOUSE_CLASSES, ignore=IGNORE_LABEL):
    """K1-lowres definition: upsample each source's heads exactly as the network would, then fuse_sources."""
    ups = [upsample_heads(m, a, out_size) for m, a in zip(mains_lr, auxs_lr)]
    return fuse_sources([u[0] for u in ups], [u[1] for u in ups], luts, policy, seg_classes, ignore)


def training_loss_lowres_and_grads(main_lr, aux_lr, labels, class_weights, alpha=20.0, dtype=torch.float32):
    """K4-lowres definition: the network's closing upsample (upsample_heads) followed by the training loss, with autograd
    through both -> (loss, d loss / d main_lr, d loss / d aux_lr)."""
    m = main_lr.detach().to(dtype).clone().requires_grad_(True)
    a = aux_lr.detach().to(dtype).clone().requires_grad_(True)
    mu, au = upsample_heads(m, a, tuple(labels.shape[-2:]))
    loss = training_loss(mu, au, labels, class_weights.to(dtype), alpha)
    gm, ga = torch.autograd.grad(loss, (m, a))
    return loss.detach(), gm, ga


def visualization_maps(main, aux):
    """The tuple branch of in_training_visualization_img, utilities/utils.py:88-97 (CPU tensors): returns
    (predictions int64 (N,H,W), heat (N,1,H,W) = -kld / max(kld) + 1)."""
    f_pred = main + 0.5 * aux
    kld = pixelwise_kld(main, aux)
    kld = (-kld / torch.max(kld).item() + 1)
    kld = torch.reshape(kld, (kld.size(0), 1, kld.size(1), kld.size(2)))
    _, predictions = torch.max(f_pred, dim=1)
    return predictions, kld


def label_to_rgb(labels, class_encoding):
    """batch_transform(labels, LongTensorToRGBPIL(class_encoding)), utilities/utils.py:157-170, 188-237, with the bytes the
    reference leaves uninitialised (labels outside the encoding) set to 0.  labels (N,H,W) int64 -> uint8 (N,3,H,W)."""
    out = torch.zeros((labels.shape[0], 3) + tuple(labels.shape[1:]), dtype=torch.uint8)
    for index, (_, color) in enumerate(class_encoding.items()):
        mask = labels == index
        for channel, value in enumerate(color):
            out[:, channel].masked_fill_(mask, value)
    return out


def cb_thresholds(label, conf, portion=0.2, ds_rate=1, seg_classes=NUM_GREENHOUSE_CLASSES, ignore=None):
    """Class-balanced (CBST/CRST-style) per-class confidence thresholds (SURVEY.md section 8 A4'').

    For class k: V_k = conf over pixels with label == k, keeping a pixel iff (row*W + col) % ds_rate == 0;
    j = floor(|V_k| * portion); thresh_k = 1.0 if j == 0 else the j-th largest element of V_k.
    `ignore` (optional): that class is never selected (apply_thresholds), so its threshold is reported as +inf instead of
    being computed; its count is still returned.
    Returns (thresh f32 (K,), n int64 (K,)) -- an exact order statistic of the given fp32 values.
    """
    label = torch.as_tensor(label)
    conf = torch.as_tensor(conf)
    h, w = label.shape[-2:]
    keep = (torch.arange(h * w) % ds_rate == 0).reshape(h, w).expand(label.shape)
    thresh = torch.ones(seg_classes, dtype=torch.float32)
    count = torch.zeros(seg_classes, dtype=torch.int64)
    for k in range(seg_classes):
        v = conf[(label == k) & keep]
        count[k] = v.numel()
        j = int(v.numel() * float(portion))
        if ignore is not None and k == ignore:
            thresh[k] = float('inf')
        elif j > 0:
            thresh[k] = torch.sort(v, descending=True).values[j - 1]
    return thresh, count


def apply_thresholds(label, conf, thresh, ignore=IGNORE_LABEL):
    """final = label if (label != ignore and conf >= thresh[label]) else ignore; mask = (final == ignore)."""
    label = torch.as_tensor(label).long()
    keep = (label != ignore) & (conf >= thresh[label])
    final = torch.where(keep, label, torch.full_like(label, ignore)).to(torch.uint8)
    return final, (final == ignore).to(torch.uint8)


# --------------------------------------------------------------------------------------------
# Synthetic inputs shared by tests, smoke() and bench.py (SURVEY.md section 8d)
# --------------------------------------------------------------------------------------------
def synthetic_logits(n, classes, h, w, seed, sigma=3.0, device='cpu'):
    """main = sigma*randn + per-image class bias; aux = main + 0.5*sigma*randn (correlated heads)."""
    g = torch.Generator(device=device).manual_seed(seed)
    main = sigma * torch.randn(n, classes, h, w, generator=g, device=device)
    bias = sigma * torch.randn(n, classes, 1, 1, generator=g, device=device)
    main = main + bias
    aux = main + 0.5 * sigma * torch.randn(n, classes, h, w, generator=g, device=device)
    return main.contiguous(), aux.contiguous()
