"""Drop-in replacements for the two hot-path modules of the reference's loss_fns/segmentation_loss.py, backed by
the CUDA kernels in libmspl_b200.so (same constructor arguments, same forward signature, same values and
gradients; CUDA tensors only)."""
import torch
from torch import nn

from .. import ops


def _upcast(x):
    """fp16 / bf16 (autocast) tensors as fp32, through a differentiable cast: autocast runs the reference's softmax and
    log_softmax in fp32, so these modules compute in fp32 and hand the gradients back in the input's dtype."""
    return x.float() if x.dtype in ops.HALF_DTYPES else x


class PixelwiseKLD(nn.Module):
    """loss_fns/segmentation_loss.py:177-189: per-pixel KL(softmax(dist1) || softmax(dist2)), (B,C,H,W)x2 -> (B,H,W),
    differentiable w.r.t. both inputs."""

    def __init__(self):
        super(PixelwiseKLD, self).__init__()

    def forward(self, dist1, dist2):
        return ops.pixelwise_kld(_upcast(dist1).contiguous(), _upcast(dist2).contiguous())


class UncertaintyWeightedSegmentationLoss(nn.Module):
    """loss_fns/segmentation_loss.py:146-175.

    Keeps the reference's construction quirk: the tensor passed as ``class_weights`` is stored as is and its
    ``ignore_idx`` entry is zeroed IN PLACE (callers reuse that tensor afterwards, uest_seg_multi_os.py:505-513).
    ``forward`` returns the mean over ALL B*H*W pixels of ``w[t] * (-log_softmax(pred)[t]) * exp(-u_weight)``.
    Unlike the reference it does not switch autograd anomaly mode on (a global, sticky debug switch at :156).
    """

    def __init__(self, num_classes, class_weights=None, ignore_idx=None, device='cuda'):
        super(UncertaintyWeightedSegmentationLoss, self).__init__()
        self.num_classes = num_classes
        self.class_weights = class_weights if class_weights is not None else torch.ones(self.num_classes).to(device)
        self.ignore_idx = ignore_idx
        if self.ignore_idx is not None:
            self.class_weights[self.ignore_idx] = 0.0

    def forward(self, pred, target, u_weight, epsilon=1e-12):   # epsilon: accepted and unused, as in the reference
        cw = self.class_weights
        if cw.dtype != torch.float32 or cw.device != pred.device:
            cw = cw.to(device=pred.device, dtype=torch.float32)
        return ops.uw_segmentation_loss(_upcast(pred).contiguous(), target.contiguous(), _upcast(u_weight), cw.contiguous())


class FusedUncertaintyWeightedLoss(nn.Module):
    """[NEW] one-launch form of the training loss expression at uest_seg_multi_os.py:1020-1023:

        kld  = PixelwiseKLD()(pred, pred_aux)
        loss = criterion(pred + 0.5*pred_aux, labels, kld) * alpha + kld.mean()

    ``forward(pred, pred_aux, labels)`` returns that loss; ``last_parts`` holds [loss, mean weighted CE, mean KLD]
    (the reference logs ``kld.mean()`` separately at :1021).  ``labels``: int64 or uint8 class indices.

    ``track_iou=True`` also folds the training loop's next statement into the launch, ``inter, union =
    miou_class.get_iou(pred, labels)`` (:1032, utilities/metrics/segmentation_miou.py:13-44 with num_classes = K): the
    per-class intersection / prediction / mask pixel counts accumulate in ``iou_counts`` ((3, K) int64, on the device, over all
    forward calls since ``reset_iou()``) without another pass over the logits or a host round trip; ``iou()`` gives what
    the loop computes from its meters at the end of the epoch, ``inter_meter.sum / (union_meter.sum + 1e-10)`` (:1049)."""

    def __init__(self, num_classes, class_weights=None, ignore_idx=None, device='cuda', alpha=20.0, track_iou=False):
        super(FusedUncertaintyWeightedLoss, self).__init__()
        self.num_classes = num_classes
        self.class_weights = class_weights if class_weights is not None else torch.ones(self.num_classes).to(device)
        self.ignore_idx = ignore_idx
        self.alpha = alpha
        self.last_parts = None
        self.track_iou = track_iou
        self.iou_counts = None
        self.iou_batches = 0
        if self.ignore_idx is not None:
            self.class_weights[self.ignore_idx] = 0.0

    def reset_iou(self):
        self.iou_counts = None
        self.iou_batches = 0

    def iou(self):
        """Per-class IoU over the batches seen since reset_iou(), as a float32 NumPy array: the loop's
        ``inter_meter.sum / (union_meter.sum + 1e-10)`` where every batch's union carries MIOU's +1e-6 (:41)."""
        import numpy as np
        if self.iou_counts is None:
            raise RuntimeError("no batch has been counted (construct with track_iou=True and call forward)")
        inter, pred, mask = (c.astype(np.float32) for c in self.iou_counts.cpu().numpy())
        union = pred + mask - inter + np.float32(self.iou_batches * 1e-6)
        return inter / (union + np.float32(1e-10))

    def _counts_for(self, pred):
        if not self.track_iou:
            return None
        if self.iou_counts is None or self.iou_counts.device != pred.device:
            self.iou_counts = torch.zeros((3, self.num_classes), dtype=torch.int64, device=pred.device)
        self.iou_batches += 1
        return self.iou_counts

    def forward(self, pred, pred_aux, labels, norm_pixels=None):
        cw = self.class_weights.to(device=pred.device, dtype=torch.float32).contiguous()
        loss, parts = ops.uw_ce_loss(pred.contiguous(), pred_aux.contiguous(), labels.contiguous(), cw, self.alpha,
                                     norm_pixels, return_parts=True, iou_counts=self._counts_for(pred))
        self.last_parts = parts
        return loss


class FusedUpsampleUncertaintyWeightedLoss(FusedUncertaintyWeightedLoss):
    """[NEW] FusedUncertaintyWeightedLoss on the tensors the network holds BEFORE its closing
    ``F.interpolate(..., size=x_size, mode='bilinear', align_corners=True)`` calls (model/segmentation/espdnet_ue.py:301-302):
    ``forward(pred_lowres, pred_aux_lowres, labels)`` equals the parent's forward on the two upsampled tensors, and the
    gradients arrive at the low-resolution tensors directly -- the upsampled logits and their gradients are never written."""

    def forward(self, pred_lowres, pred_aux_lowres, labels, norm_pixels=None):
        if self.track_iou:
            raise NotImplementedError("track_iou needs the full-resolution main logits; use FusedUncertaintyWeightedLoss")
        cw = self.class_weights.to(device=pred_lowres.device, dtype=torch.float32).contiguous()
        loss, parts = ops.uw_ce_loss_lowres(pred_lowres.contiguous(), pred_aux_lowres.contiguous(), labels.contiguous(), cw,
                                            self.alpha, norm_pixels, return_parts=True)
        self.last_parts = parts
        return loss


class NIDLoss(nn.Module):
    """loss_fns/segmentation_loss.py:54-118: normalised information distance between the grey-scale camera image and the
    soft-argmax label map, rescaled as ``(nid - 0.95) * 20`` -- the optional ``--use-nid`` training term
    (uest_seg_multi_os.py:514, 1027-1030).  Same constructor and ``forward(camera, label)``; one fused pass per direction."""

    def __init__(self, image_bin=16, label_bin=4, bw_camera=0.005, bw_label=0.001):
        super(NIDLoss, self).__init__()
        self.K = image_bin
        self.C = label_bin
        self.bw_camera = bw_camera
        self.bw_label = bw_label

    def forward(self, camera, label):
        return ops.nid_loss(camera, label, self.K, self.C, self.bw_camera, self.bw_label)
