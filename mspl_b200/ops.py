"""Tensor-in / tensor-out entry points over libmspl_b200.so (no NumPy, no host sync, no CPU fallback).

These are the batched fast paths behind the reference-named callables in ``mspl_b200.uest_seg_multi_os`` and
``mspl_b200.loss_fns.segmentation_loss``.  Every function enqueues on the current CUDA stream of the tensors'
device and returns device tensors.
"""
import ctypes
from collections import namedtuple

import numpy as np
import torch

from . import _lib

RADIX_BINS = 2048
RADIX_PASSES = 3
MAX_SOURCES = 8
MAX_CLASSES = 8
POLICY_VOTE, POLICY_PROB = 0, 1

FuseResult = namedtuple("FuseResult", "label conf unc kld class_hist conf_hist marginal")


def _require_cuda(t, name, dtype=None, ndim=None):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor, got %s" % (name, type(t).__name__))
    if not t.is_cuda:
        raise ValueError("%s must be a CUDA tensor (mspl_b200 has no CPU path), got device %s" % (name, t.device))
    if dtype is not None and t.dtype != dtype:
        raise ValueError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if ndim is not None and t.dim() != ndim:
        raise ValueError("%s must have %d dims, got shape %s" % (name, ndim, tuple(t.shape)))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    return t


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def vote_threshold(num_sources, thresh=None):
    """merge_outputs' threshold rule (uest_seg_multi_os.py:697-705): None/'half'/invalid -> S//2+1,
    'all' -> S, an int <= S -> itself."""
    if thresh is None or (isinstance(thresh, str) and thresh == 'half'):
        return num_sources // 2 + 1
    if isinstance(thresh, str) and thresh == 'all':
        return num_sources
    if isinstance(thresh, int) and thresh <= num_sources:       # bool included, as the reference's isinstance(thresh, int)
        return int(thresh)
    return num_sources // 2 + 1


def _lut_bytes(lut, num_src_classes, num_classes):
    arr = np.asarray(lut.cpu() if isinstance(lut, torch.Tensor) else lut).astype(np.int64).reshape(-1)
    if arr.size != num_src_classes:
        raise ValueError("label table has %d entries for a %d-class source" % (arr.size, num_src_classes))
    if arr.min() < 0 or arr.max() >= num_classes:
        raise ValueError("label table values must lie in [0, %d)" % num_classes)
    return (ctypes.c_ubyte * arr.size)(*arr.tolist())


def fuse_sources(mains, auxs, luts, policy='half', num_classes=5, ignore_label=4, ds_rate=1,
                 want_conf=True, want_unc=True, want_kld=False, want_conf_hist=True, count_marginal=True,
                 class_hist=None, conf_hist=None, marginal=None, label_out=None, conf_out=None, unc_out=None):
    """K1: fused multi-source pseudo-label generation (replaces uest_seg_multi_os.py:897-921).

    mains/auxs: lists (one entry per source) of (N, C_s, H, W) fp32 CUDA logits; luts: per-source tables
    source class -> target class.  policy: 'half' | 'all' | int (the reference's vote, merge_outputs) or
    'prob' ([NEW] averaged greenhouse-class probabilities).  Histogram / counter tensors passed in are
    accumulated into (int64); otherwise fresh zeroed ones are returned.  label_out/conf_out/unc_out: optional
    preallocated (N,H,W) outputs (e.g. slices of a dataset-wide map).
    """
    S = len(mains)
    if S < 1 or S > MAX_SOURCES or len(auxs) != S or len(luts) != S:
        raise ValueError("need 1..%d sources with matching mains/auxs/luts" % MAX_SOURCES)
    if not (2 <= num_classes <= MAX_CLASSES) or not (0 <= ignore_label < num_classes):
        raise ValueError("num_classes must be in [2,%d] and ignore_label inside it" % MAX_CLASSES)
    m0 = _require_cuda(mains[0], "mains[0]", torch.float32, 4)
    n, _, h, w = m0.shape
    dev = m0.device
    lut_bufs, cls = [], []
    for s in range(S):
        m = _require_cuda(mains[s], "mains[%d]" % s, torch.float32, 4)
        a = _require_cuda(auxs[s], "auxs[%d]" % s, torch.float32, 4)
        if m.shape != a.shape or m.shape[0] != n or m.shape[2:] != (h, w) or m.device != dev or a.device != dev:
            raise ValueError("source %d: main/aux shapes or devices disagree" % s)
        cls.append(m.shape[1])
        lut_bufs.append(_lut_bytes(luts[s], m.shape[1], num_classes))
    if policy == 'prob':
        pol, vt = POLICY_PROB, 0
    else:
        pol, vt = POLICY_VOTE, vote_threshold(S, policy)
    hw = h * w
    def _out(t, name, dtype, wanted):
        if t is not None:
            if _require_cuda(t, name, dtype).shape != (n, h, w) or t.device != dev:
                raise ValueError("%s must be a (%d,%d,%d) tensor on %s" % (name, n, h, w, dev))
            return t
        return torch.empty((n, h, w), dtype=dtype, device=dev) if wanted else None

    label = _out(label_out, "label_out", torch.uint8, True)
    conf = _out(conf_out, "conf_out", torch.float32, want_conf or want_conf_hist)
    unc = _out(unc_out, "unc_out", torch.float32, want_unc)
    kld = [torch.empty((n, h, w), dtype=torch.float32, device=dev) for _ in range(S)] if want_kld else None
    if class_hist is None:
        class_hist = torch.zeros(num_classes, dtype=torch.int64, device=dev)
    if want_conf_hist and conf_hist is None:
        conf_hist = torch.zeros((num_classes, RADIX_BINS), dtype=torch.int64, device=dev)
    if count_marginal and marginal is None:
        marginal = torch.zeros((), dtype=torch.int64, device=dev)
    for t, nm in ((class_hist, "class_hist"), (conf_hist, "conf_hist"), (marginal, "marginal")):
        if t is not None:
            _require_cuda(t, nm, torch.int64)
    vp = ctypes.c_void_p
    main_ptrs = (vp * S)(*[m.data_ptr() for m in mains])
    aux_ptrs = (vp * S)(*[a.data_ptr() for a in auxs])
    kld_ptrs = (vp * S)(*[k.data_ptr() for k in kld]) if kld is not None else None
    ncls = (ctypes.c_int * S)(*cls)
    lut_ptrs = (vp * S)(*[ctypes.addressof(b) for b in lut_bufs])
    lib = _lib.load()
    if n == 0:      # nothing to label: empty maps, untouched histograms
        return FuseResult(label, conf, unc, kld, class_hist, conf_hist if want_conf_hist else None,
                          marginal if count_marginal else None)
    with torch.cuda.device(dev):
        st = lib.mspl_fuse_sources(S, main_ptrs, aux_ptrs, ncls, lut_ptrs, n, hw, num_classes, pol, vt,
                                   ignore_label, int(ds_rate), _ptr(label), _ptr(conf), _ptr(unc), kld_ptrs,
                                   _ptr(class_hist), _ptr(conf_hist if want_conf_hist else None),
                                   _ptr(marginal if count_marginal else None), _stream(dev))
    _lib.check(st, "mspl_fuse_sources")
    return FuseResult(label, conf, unc, kld, class_hist, conf_hist if want_conf_hist else None,
                      marginal if count_marginal else None)


def fuse_sources_lowres(mains, auxs, luts, out_size, policy='half', num_classes=5, ignore_label=4, ds_rate=1,
                        want_conf=True, want_unc=True, want_kld=False, want_conf_hist=True, count_marginal=True,
                        class_hist=None, conf_hist=None, marginal=None, label_out=None, conf_out=None, unc_out=None):
    """K1 with the networks' final bilinear upsample fused in: mains[s] is (N, C_s, hm, wm), auxs[s] is (N, C_s, ha, wa) --
    the tensors ESPDNetUE feeds to its closing ``F.interpolate(..., size=out_size, mode='bilinear', align_corners=True)``
    (model/segmentation/espdnet_ue.py:301-302) -- and the labels come out at ``out_size = (H, W)``.  Everything else is as
    in fuse_sources.  Raises NotImplementedError when the geometry is not supported by the fused kernel (row lengths not
    multiples of 4, H*W % 4 != 0, or source rows too wide for shared memory): upsample and call fuse_sources then."""
    S = len(mains)
    if S < 1 or S > MAX_SOURCES or len(auxs) != S or len(luts) != S:
        raise ValueError("need 1..%d sources with matching mains/auxs/luts" % MAX_SOURCES)
    if not (2 <= num_classes <= MAX_CLASSES) or not (0 <= ignore_label < num_classes):
        raise ValueError("num_classes must be in [2,%d] and ignore_label inside it" % MAX_CLASSES)
    h, w = int(out_size[0]), int(out_size[1])
    m0 = _require_cuda(mains[0], "mains[0]", torch.float32, 4)
    n, dev = m0.shape[0], m0.device
    lut_bufs, cls, mhw, ahw = [], [], [], []
    for s in range(S):
        m = _require_cuda(mains[s], "mains[%d]" % s, torch.float32, 4)
        a = _require_cuda(auxs[s], "auxs[%d]" % s, torch.float32, 4)
        if m.shape[:2] != a.shape[:2] or m.shape[0] != n or m.device != dev or a.device != dev:
            raise ValueError("source %d: main/aux batch, class count or device disagree" % s)
        cls.append(m.shape[1])
        mhw += [m.shape[2], m.shape[3]]
        ahw += [a.shape[2], a.shape[3]]
        lut_bufs.append(_lut_bytes(luts[s], m.shape[1], num_classes))
    if policy == 'prob':
        pol, vt = POLICY_PROB, 0
    else:
        pol, vt = POLICY_VOTE, vote_threshold(S, policy)
    def _out(t, name, dtype, wanted):
        if t is not None:
            if _require_cuda(t, name, dtype).shape != (n, h, w) or t.device != dev:
                raise ValueError("%s must be a (%d,%d,%d) tensor on %s" % (name, n, h, w, dev))
            return t
        return torch.empty((n, h, w), dtype=dtype, device=dev) if wanted else None

    label = _out(label_out, "label_out", torch.uint8, True)
    conf = _out(conf_out, "conf_out", torch.float32, want_conf or want_conf_hist)
    unc = _out(unc_out, "unc_out", torch.float32, want_unc)
    kld = [torch.empty((n, h, w), dtype=torch.float32, device=dev) for _ in range(S)] if want_kld else None
    if class_hist is None:
        class_hist = torch.zeros(num_classes, dtype=torch.int64, device=dev)
    if want_conf_hist and conf_hist is None:
        conf_hist = torch.zeros((num_classes, RADIX_BINS), dtype=torch.int64, device=dev)
    if count_marginal and marginal is None:
        marginal = torch.zeros((), dtype=torch.int64, device=dev)
    for t, nm in ((class_hist, "class_hist"), (conf_hist, "conf_hist"), (marginal, "marginal")):
        if t is not None:
            _require_cuda(t, nm, torch.int64)
    vp = ctypes.c_void_p
    main_ptrs = (vp * S)(*[m.data_ptr() for m in mains])
    aux_ptrs = (vp * S)(*[a.data_ptr() for a in auxs])
    kld_ptrs = (vp * S)(*[k.data_ptr() for k in kld]) if kld is not None else None
    ncls = (ctypes.c_int * S)(*cls)
    lut_ptrs = (vp * S)(*[ctypes.addressof(b) for b in lut_bufs])
    mhw_arr, ahw_arr = (ctypes.c_int * (2 * S))(*mhw), (ctypes.c_int * (2 * S))(*ahw)
    if n == 0:
        return FuseResult(label, conf, unc, kld, class_hist, conf_hist if want_conf_hist else None,
                          marginal if count_marginal else None)
    with torch.cuda.device(dev):
        st = _lib.load().mspl_fuse_sources_lowres(S, main_ptrs, aux_ptrs, ncls, lut_ptrs, mhw_arr, ahw_arr, n, h, w, num_classes,
                                                  pol, vt, ignore_label, int(ds_rate), _ptr(label), _ptr(conf), _ptr(unc), kld_ptrs,
                                                  _ptr(class_hist), _ptr(conf_hist if want_conf_hist else None),
                                                  _ptr(marginal if count_marginal else None), _stream(dev))
    if st == -3:
        raise NotImplementedError("fuse_sources_lowres: geometry not supported by the fused-upsample kernel; upsample and use "
                                  "fuse_sources")
    _lib.check(st, "mspl_fuse_sources_lowres")
    return FuseResult(label, conf, unc, kld, class_hist, conf_hist if want_conf_hist else None,
                      marginal if count_marginal else None)


def vote_labels(labels, num_classes=5, thresh=None, ignore_label=4):
    """merge_outputs on a (S, ...) uint8 CUDA tensor of hard labels -> uint8 tensor of shape labels.shape[1:]."""
    labels = _require_cuda(labels, "labels", torch.uint8)
    S = labels.shape[0]
    out = torch.empty(labels.shape[1:], dtype=torch.uint8, device=labels.device)
    npix = out.numel()
    with torch.cuda.device(labels.device):
        st = _lib.load().mspl_vote_labels(_ptr(labels), S, npix, num_classes, vote_threshold(S, thresh), ignore_label,
                                          _ptr(out), _stream(labels.device))
    _lib.check(st, "mspl_vote_labels")
    return out


def softmax_kld(main, aux, want_prob=True, want_kld=True):
    """K0: (softmax(main + 0.5*aux) over classes, KL(softmax(main)||softmax(aux))) for (N,C,H,W) logits."""
    main = _require_cuda(main, "main", torch.float32, 4)
    aux = _require_cuda(aux, "aux", torch.float32, 4)
    if main.shape != aux.shape:
        raise ValueError("main/aux shapes differ")
    n, c, h, w = main.shape
    prob = torch.empty_like(main) if want_prob else None
    kld = torch.empty((n, h, w), dtype=torch.float32, device=main.device) if want_kld else None
    with torch.cuda.device(main.device):
        st = _lib.load().mspl_softmax_kld(_ptr(main), _ptr(aux), n, c, h * w, _ptr(prob), _ptr(kld), _stream(main.device))
    _lib.check(st, "mspl_softmax_kld")
    return prob, kld


def select_and_apply(label, conf, portion=0.2, ds_rate=1, num_classes=5, ignore_label=4, conf_hist=None, all_reduce=None,
                     want_final=True, want_mask=False, final_hist=None, hist_reduced=False):
    """K2+K3, bracketed protocol: class-balanced thresholds AND the thresholded label map in ONE pass over (label, conf).

    label (N,H,W) u8, conf (N,H,W) f32.  conf_hist: the linear confidence histogram already accumulated by fuse_sources
    (consumed: zeroed on return); if None it is computed here (one more 5 B/pixel pass).
    all_reduce: None for a single rank -- the candidate passes, their selects and the patch then run as ONE launch
    (mspl_cand_resolve) -- or a callable applied in place to an int64 tensor (``lambda t: dist.all_reduce(t)``): every rank
    then selects the same bins, thresholds are identical for 1 or N GPUs and the returned final_hist is the GLOBAL one on every
    rank (derived from the all-reduced histograms, no collective of its own when ds_rate == 1).  hist_reduced: conf_hist has
    already been all-reduced by the caller (the pipeline packs it with the other statistics into one collective).
    No host synchronisation.  The ignore class is never selected, so its threshold is not resolved: thresh[ignore_label] = +inf
    (kept_count[ignore_label] is still its pixel count).  ignore_label=None resolves every class; no map can be written then.
    Returns (thresh f32 (K,), kept_count i64 (K,), final u8 or None, mask u8 or None, final_hist i64 (K,) or None)."""
    label = _require_cuda(label, "label", torch.uint8)
    conf = _require_cuda(conf, "conf", torch.float32)
    if label.shape != conf.shape or label.dim() < 2:
        raise ValueError("label/conf must share a (..., H, W) shape")
    dev = label.device
    hw = label.shape[-1] * label.shape[-2]
    npix = label.numel()
    if npix >= 2 ** 32:
        raise NotImplementedError("select_and_apply indexes candidates with 32 bits; use cb_thresholds_radix + apply_thresholds")
    lib = _lib.load()
    K = num_classes
    state = torch.zeros(lib.mspl_radix_state_bytes(K), dtype=torch.uint8, device=dev)
    thresh = torch.empty(K, dtype=torch.float32, device=dev)
    bracket = torch.empty((K, 2), dtype=torch.float32, device=dev)
    kept = torch.zeros(K, dtype=torch.int64, device=dev)
    cand_index = torch.empty(max(npix, 1), dtype=torch.int32, device=dev)      # u32 indices; worst case every pixel is a candidate
    cand_count = torch.zeros((), dtype=torch.int64, device=dev)
    outputs = want_final or want_mask or final_hist is not None
    if ignore_label is None:
        if outputs:
            raise ValueError("a label map / mask / final histogram needs an ignore_label")
        ign = -1
    else:
        ign = int(ignore_label)
    final = torch.empty_like(label) if want_final else None
    mask = torch.empty_like(label) if want_mask else None
    if outputs and final_hist is None:
        final_hist = torch.zeros(K, dtype=torch.int64, device=dev)
    hist = conf_hist
    if hist is not None:
        _require_cuda(hist, "conf_hist", torch.int64)
    else:
        hist = torch.zeros((K, RADIX_BINS), dtype=torch.int64, device=dev)
    single = all_reduce is None
    with torch.cuda.device(dev):
        st = _stream(dev)
        if conf_hist is None:
            _lib.check(lib.mspl_conf_hist(_ptr(label), _ptr(conf), npix, hw, K, _ptr(hist), int(ds_rate), st), "mspl_conf_hist")
        if not single and not (hist_reduced and conf_hist is not None):
            all_reduce(hist)
        # with ds_rate 1 the histogram covers every pixel, so the final class counts are read off it (of all ranks' pixels once
        # it is all-reduced) instead of being counted per pixel by the classify pass
        from_hist = outputs and int(ds_rate) == 1
        _lib.check(lib.mspl_bracket_select(_ptr(hist), K, float(portion), ign, _ptr(state), _ptr(bracket), _ptr(thresh), _ptr(kept),
                                           None, _ptr(final_hist if from_hist else None), st), "mspl_bracket_select")
        _lib.check(lib.mspl_bracket_classify(_ptr(label), _ptr(conf), _ptr(bracket), npix, K, ign, _ptr(final), _ptr(mask),
                                             _ptr(final_hist if outputs and not from_hist else None), _ptr(cand_index),
                                             _ptr(cand_count), st), "mspl_bracket_classify")
        resolved = False
        if single:
            rc = lib.mspl_cand_resolve(_ptr(label), _ptr(conf), _ptr(cand_index), _ptr(cand_count), hw, K, ign, int(ds_rate),
                                       _ptr(state), _ptr(thresh), _ptr(final), _ptr(mask), _ptr(final_hist if outputs else None), st)
            if rc != -3:        # MSPL_ERR_UNSUPPORTED: no room for an 8-CTA cluster on this device -> the multi-launch passes below
                _lib.check(rc, "mspl_cand_resolve")
                resolved = True
            all_reduce = lambda t: t
        if not resolved:
            for p in range(RADIX_PASSES):
                _lib.check(lib.mspl_cand_hist_pass(_ptr(label), _ptr(conf), _ptr(cand_index), _ptr(cand_count), hw, K, p, _ptr(state),
                                                   _ptr(hist), int(ds_rate), st), "mspl_cand_hist_pass")
                all_reduce(hist)
                _lib.check(lib.mspl_cand_select(_ptr(hist), K, p, _ptr(state), _ptr(thresh), _ptr(final_hist if from_hist else None),
                                                ign, st), "mspl_cand_select")
            if outputs:
                _lib.check(lib.mspl_cand_apply(_ptr(label), _ptr(conf), _ptr(thresh), _ptr(cand_index), _ptr(cand_count), K, ign,
                                               _ptr(final), _ptr(mask), _ptr(None if from_hist else final_hist), st), "mspl_cand_apply")
                if not from_hist:
                    all_reduce(final_hist)      # ds_rate > 1: the classify pass counted this rank's pixels only
    return thresh, kept, final, mask, (final_hist if outputs else None)


# kernels select_and_apply launches: single rank = bracket_select + classify + cand_resolve; with an all-reduce between the
# passes = bracket_select + classify + 3 x (cand_hist + cand_select) + cand_apply
SELECT_AND_APPLY_LAUNCHES = 3
SELECT_AND_APPLY_LAUNCHES_SHARDED = 9


def new_label_stats(num_classes, device):
    """One int64 buffer holding every statistic K1 accumulates, so that N ranks exchange them in ONE all-reduce:
    returns (buffer, conf_hist (K, 2048) view, class_hist (K,) view, marginal () view)."""
    K = num_classes
    buf = torch.zeros(K * RADIX_BINS + K + 1, dtype=torch.int64, device=device)
    return buf, buf[:K * RADIX_BINS].view(K, RADIX_BINS), buf[K * RADIX_BINS:K * RADIX_BINS + K], buf[K * RADIX_BINS + K:].view(())


def cb_thresholds(label, conf, portion=0.2, ds_rate=1, num_classes=5, conf_hist=None, all_reduce=None, ignore_label=None):
    """K2: class-balanced thresholds only (bracketed protocol without writing a label map); see select_and_apply.
    ignore_label=None resolves the threshold of every class (the definition of the oracle's cb_thresholds); naming the
    ignore class skips it (thresh = +inf), which is much cheaper when its pixels all share conf == 0 (vote policies).
    Returns (thresh f32 (K,), kept_count int64 (K,))."""
    thresh, kept, _, _, _ = select_and_apply(label, conf, portion, ds_rate, num_classes, ignore_label=ignore_label,
                                             conf_hist=conf_hist, all_reduce=all_reduce, want_final=False, want_mask=False)
    return thresh, kept


def cb_thresholds_radix(label, conf, portion=0.2, ds_rate=1, num_classes=5, all_reduce=None):
    """K2, generic protocol: 3 full radix passes over the order-preserving key of conf (no linear histogram, no candidate
    list).  Same definition and the same bits as cb_thresholds; 15 B/pixel instead of 5-6."""
    label = _require_cuda(label, "label", torch.uint8)
    conf = _require_cuda(conf, "conf", torch.float32)
    if label.shape != conf.shape or label.dim() < 2:
        raise ValueError("label/conf must share a (..., H, W) shape")
    dev = label.device
    hw = label.shape[-1] * label.shape[-2]
    npix = label.numel()
    lib = _lib.load()
    K = num_classes
    state = torch.zeros(lib.mspl_radix_state_bytes(K), dtype=torch.uint8, device=dev)
    thresh = torch.empty(K, dtype=torch.float32, device=dev)
    kept = torch.zeros(K, dtype=torch.int64, device=dev)
    hist = torch.zeros((K, RADIX_BINS), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        st = _stream(dev)
        for p in range(RADIX_PASSES):
            _lib.check(lib.mspl_radix_hist_pass(_ptr(label), _ptr(conf), npix, hw, K, p, _ptr(state), _ptr(hist),
                                                int(ds_rate), st), "mspl_radix_hist_pass")
            if all_reduce is not None:
                all_reduce(hist)
            _lib.check(lib.mspl_radix_select(_ptr(hist), K, p, float(portion), _ptr(state), _ptr(thresh), _ptr(kept), st),
                       "mspl_radix_select")
    return thresh, kept


def apply_thresholds(label, conf, thresh, ignore_label=4, want_mask=True, final_hist=None):
    """K3: final = label if (label != ignore and conf >= thresh[label]) else ignore; mask = (final == ignore).
    Returns (final u8, mask u8 or None, final_hist int64 (K,))."""
    label = _require_cuda(label, "label", torch.uint8)
    conf = _require_cuda(conf, "conf", torch.float32)
    thresh = _require_cuda(thresh, "thresh", torch.float32, 1)
    dev = label.device
    K = thresh.numel()
    final = torch.empty_like(label)
    mask = torch.empty_like(label) if want_mask else None
    if final_hist is None:
        final_hist = torch.zeros(K, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        st = _lib.load().mspl_apply_thresholds(_ptr(label), _ptr(conf), _ptr(thresh), label.numel(), K, ignore_label,
                                               _ptr(final), _ptr(mask), _ptr(final_hist), _stream(dev))
    _lib.check(st, "mspl_apply_thresholds")
    return final, mask, final_hist


# ---- loss ---------------------------------------------------------------------------------------------------
_workspaces = {}


def _workspace(dev):
    """One zeroed reduction workspace per (device, stream): kernels leave it zeroed for the next call."""
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None:
        ws = torch.zeros(_lib.load().mspl_uw_ce_workspace_bytes(), dtype=torch.uint8, device=dev)
        _workspaces[key] = ws
    return ws


def _class_index_target(target):
    """Targets of the fused losses: int64 (the reference's format, what torch.gather needs) or uint8 (the format the label
    maps are generated, stored and saved in -- 1 byte per pixel of HBM traffic instead of 8).  Returns (tensor, is_u8)."""
    if isinstance(target, torch.Tensor) and target.dtype == torch.uint8:
        return _require_cuda(target, "target", torch.uint8, 3), True
    return _require_cuda(target, "target", torch.int64, 3), False


# fp16 / bf16 logits of K4 (mspl_uw_ce_step_half): torch dtype -> MSPL_DTYPE_F16 / MSPL_DTYPE_BF16
HALF_DTYPES = {torch.float16: 1, torch.bfloat16: 2}


def uw_ce_fwd_bwd(main, aux, target, class_weights, alpha=20.0, norm_pixels=None, grad_scale=1.0, backward=True, iou_counts=None,
                  grad_scale_dev=None):
    """K4, explicit form: returns (out3, d_main, d_aux) with out3 = [loss, mean w*ce*exp(-kld), mean kld] on device and
    the gradients of loss*grad_scale (None, None when backward=False).  target: (N,H,W) class indices, int64 or uint8.
    iou_counts: optional (3, K) int64 CUDA tensor that the same launch ADDS the MIOU.get_iou(main, target) pixel counts to
    ([intersection | prediction | mask] per class, utilities/metrics/segmentation_miou.py:13-44 with num_classes = K).

    main/aux may also both be fp16 or both bf16 (autocast logits): the kernel upcasts them exactly and computes in fp32, out3
    stays fp32 and the gradients come back in the logits' dtype, scaled by grad_scale (and, for these dtypes only, by the
    device scalar grad_scale_dev, a 1-element fp32 tensor) before they are rounded."""
    half = isinstance(main, torch.Tensor) and main.dtype in HALF_DTYPES
    main = _require_cuda(main, "main", main.dtype if half else torch.float32, 4)
    aux = _require_cuda(aux, "aux", main.dtype, 4)
    target, u8 = _class_index_target(target)
    cw = _require_cuda(class_weights, "class_weights", torch.float32, 1)
    n, k, h, w = main.shape
    if aux.shape != main.shape or target.shape != (n, h, w) or cw.numel() != k:
        raise ValueError("shape mismatch: main %s aux %s target %s class_weights %s" %
                         (tuple(main.shape), tuple(aux.shape), tuple(target.shape), tuple(cw.shape)))
    if k > MAX_CLASSES:
        raise NotImplementedError("fused loss supports up to %d classes; use PixelwiseKLD + "
                                  "UncertaintyWeightedSegmentationLoss modules for %d" % (MAX_CLASSES, k))
    if grad_scale_dev is not None:
        if not half:
            raise ValueError("grad_scale_dev applies to fp16 / bf16 logits; scale fp32 gradients with grad_scale")
        _require_cuda(grad_scale_dev, "grad_scale_dev", torch.float32)
        if grad_scale_dev.numel() != 1:
            raise ValueError("grad_scale_dev must hold one value")
    dev = main.device
    out3 = torch.empty(3, dtype=torch.float32, device=dev)
    d_main = torch.empty_like(main) if backward else None
    d_aux = torch.empty_like(aux) if backward else None
    ws = _workspace(dev)
    norm = float(norm_pixels) if norm_pixels is not None else float(n * h * w)
    if iou_counts is not None:
        iou_counts = _require_cuda(iou_counts, "iou_counts", torch.int64, 2)
        if iou_counts.shape != (3, k) or iou_counts.device != dev:
            raise ValueError("iou_counts must be a (3, %d) int64 tensor on %s" % (k, dev))
    with torch.cuda.device(dev):
        if half:
            st = _lib.load().mspl_uw_ce_step_half(_ptr(main), _ptr(aux), HALF_DTYPES[main.dtype], _ptr(target), int(u8), _ptr(cw), n,
                                                  k, h * w, float(alpha), norm, float(grad_scale), _ptr(grad_scale_dev), _ptr(out3),
                                                  _ptr(d_main), _ptr(d_aux), _ptr(iou_counts), _ptr(ws), ws.numel(), _stream(dev))
        else:
            st = _lib.load().mspl_uw_ce_step(_ptr(main), _ptr(aux), _ptr(target), int(u8), _ptr(cw), n, k, h * w, float(alpha), norm,
                                             float(grad_scale), _ptr(out3), _ptr(d_main), _ptr(d_aux), _ptr(iou_counts), _ptr(ws),
                                             ws.numel(), _stream(dev))
    _lib.check(st, "mspl_uw_ce_step_half" if half else "mspl_uw_ce_step")
    return out3, d_main, d_aux


class _UwCeLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, main, aux, target, class_weights, alpha, norm_pixels, iou_counts=None):
        need = main.requires_grad or aux.requires_grad
        ctx.deferred = main.dtype in HALF_DTYPES and need
        if ctx.deferred:
            # fp16 / bf16: the gradients must be scaled by the upstream gradient (a GradScaler's loss scale) before they are
            # rounded, and that scale is only known in backward.  So this launch is forward-only, and backward runs K4 once more
            # with the upstream gradient as its device scale.
            out3, _, _ = uw_ce_fwd_bwd(main.detach(), aux.detach(), target, class_weights.detach(), alpha, norm_pixels,
                                       backward=False, iou_counts=iou_counts)
            ctx.save_for_backward(main, aux, target, class_weights)
            ctx.cfg = (alpha, norm_pixels)
            ctx.grads = None
        else:
            out3, d_main, d_aux = uw_ce_fwd_bwd(main.detach(), aux.detach(), target, class_weights.detach(), alpha, norm_pixels,
                                                1.0, backward=need, iou_counts=iou_counts)
            ctx.grads = (d_main, d_aux)
        ctx.mark_non_differentiable(out3)
        return out3[0].clone(), out3

    @staticmethod
    def backward(ctx, grad_loss, _grad_parts):
        if getattr(ctx, "deferred", False):
            main, aux, target, cw = ctx.saved_tensors
            g = grad_loss.detach().to(torch.float32).reshape(1).contiguous()
            _, d_main, d_aux = uw_ce_fwd_bwd(main.detach(), aux.detach(), target, cw.detach(), *ctx.cfg, grad_scale_dev=g)
            return d_main, d_aux, None, None, None, None, None
        if ctx.grads is None:
            raise RuntimeError("uw_ce_loss: backward through this loss a second time is not supported (its gradients are "
                               "produced by the forward launch and handed over once)")
        d_main, d_aux = ctx.grads
        ctx.grads = None
        if d_main is None:
            return (None,) * 7
        # upstream gradient applied on device, skipped inside the kernel when it is exactly 1 (loss.backward())
        g = grad_loss.detach().to(torch.float32).reshape(1).contiguous()
        lib = _lib.load()
        with torch.cuda.device(d_main.device):
            st = _stream(d_main.device)
            _lib.check(lib.mspl_scale_inplace(_ptr(d_main), d_main.numel(), _ptr(g), st), "mspl_scale_inplace")
            _lib.check(lib.mspl_scale_inplace(_ptr(d_aux), d_aux.numel(), _ptr(g), st), "mspl_scale_inplace")
        return d_main, d_aux, None, None, None, None, None


def uw_ce_loss(main, aux, target, class_weights, alpha=20.0, norm_pixels=None, return_parts=False, iou_counts=None):
    """K4 with autograd: the value of ``criterion(main + 0.5*aux, target, kld) * alpha + kld.mean()`` with
    ``kld = PixelwiseKLD()(main, aux)`` (uest_seg_multi_os.py:1020-1023), forward and backward in ONE kernel launch.
    norm_pixels overrides the divisor of the means (global pixel count under data parallelism); iou_counts: see
    uw_ce_fwd_bwd (the training loop's ``miou_class.get_iou(pred, labels)`` of :1032 counted by the same launch).
    fp16 / bf16 logits (autocast) take one forward-only launch here and one forward+backward launch in backward, which scales
    the gradients by the upstream gradient before rounding them to the logits' dtype."""
    loss, parts = _UwCeLoss.apply(main, aux, target, class_weights, alpha, norm_pixels, iou_counts)
    return (loss, parts) if return_parts else loss


def uw_ce_lowres_fwd_bwd(main_lr, aux_lr, target, class_weights, alpha=20.0, norm_pixels=None, grad_scale=1.0, backward=True):
    """K4-lowres, explicit form: main_lr (N,K,hm,wm), aux_lr (N,K,ha,wa) are the tensors the network feeds to its closing
    bilinear align_corners=True upsample (model/segmentation/espdnet_ue.py:301-302), target (N,H,W) int64 or uint8 gives the
    output size.  Returns (out3, d_main_lr, d_aux_lr) like uw_ce_fwd_bwd, the gradients being w.r.t. the PRE-upsample tensors."""
    main_lr = _require_cuda(main_lr, "main_lr", torch.float32, 4)
    aux_lr = _require_cuda(aux_lr, "aux_lr", torch.float32, 4)
    target, u8 = _class_index_target(target)
    cw = _require_cuda(class_weights, "class_weights", torch.float32, 1)
    n, k, hm, wm = main_lr.shape
    ha, wa = aux_lr.shape[2:]
    h, w = target.shape[1:]
    if aux_lr.shape[:2] != (n, k) or target.shape[0] != n or cw.numel() != k:
        raise ValueError("shape mismatch: main %s aux %s target %s class_weights %s" %
                         (tuple(main_lr.shape), tuple(aux_lr.shape), tuple(target.shape), tuple(cw.shape)))
    dev = main_lr.device
    out3 = torch.empty(3, dtype=torch.float32, device=dev)
    d_main = torch.empty_like(main_lr) if backward else None
    d_aux = torch.empty_like(aux_lr) if backward else None
    ws = _workspace(dev)
    norm = float(norm_pixels) if norm_pixels is not None else float(n * h * w)
    lib = _lib.load()
    entry = lib.mspl_uw_ce_lowres_fwd_bwd_u8 if u8 else lib.mspl_uw_ce_lowres_fwd_bwd
    with torch.cuda.device(dev):
        st = entry(_ptr(main_lr), _ptr(aux_lr), _ptr(target), _ptr(cw), n, k, hm, wm, ha, wa, h, w, float(alpha), norm,
                   float(grad_scale), _ptr(out3), _ptr(d_main), _ptr(d_aux), _ptr(ws), ws.numel(), _stream(dev))
    if st == -3:
        raise NotImplementedError("uw_ce_lowres: geometry not supported by the fused-upsample loss kernel (more than %d classes, "
                                  "a source larger than the output, or rows too wide for shared memory); upsample and use "
                                  "uw_ce_loss" % MAX_CLASSES)
    _lib.check(st, "mspl_uw_ce_lowres_fwd_bwd_u8" if u8 else "mspl_uw_ce_lowres_fwd_bwd")
    return out3, d_main, d_aux


class _UwCeLossLowres(torch.autograd.Function):
    @staticmethod
    def forward(ctx, main_lr, aux_lr, target, class_weights, alpha, norm_pixels, _reserved=None):   # 7 inputs like _UwCeLoss
        need = main_lr.requires_grad or aux_lr.requires_grad
        out3, d_main, d_aux = uw_ce_lowres_fwd_bwd(main_lr.detach(), aux_lr.detach(), target, class_weights.detach(), alpha,
                                                   norm_pixels, 1.0, backward=need)
        ctx.grads = (d_main, d_aux)
        ctx.mark_non_differentiable(out3)
        return out3[0].clone(), out3

    backward = _UwCeLoss.backward          # same hand-over of the gradients produced by the forward launch


def uw_ce_loss_lowres(main_lr, aux_lr, target, class_weights, alpha=20.0, norm_pixels=None, return_parts=False):
    """K4-lowres with autograd: the training loss of uest_seg_multi_os.py:1020-1023 evaluated on
    ``F.interpolate(main_lr, target.shape[1:], mode='bilinear', align_corners=True)`` (and the same for aux_lr) without ever
    materialising the upsampled logits or their gradients; forward, backward and both interpolation transposes in ONE launch."""
    loss, parts = _UwCeLossLowres.apply(main_lr, aux_lr, target, class_weights, alpha, norm_pixels, None)
    return (loss, parts) if return_parts else loss


def kld_fwd(d1, d2):
    return softmax_kld(d1, d2, want_prob=False, want_kld=True)[1]


class _PixelwiseKLD(torch.autograd.Function):
    @staticmethod
    def forward(ctx, d1, d2):
        d1c, d2c = d1.detach().contiguous(), d2.detach().contiguous()
        ctx.save_for_backward(d1c, d2c)
        return kld_fwd(d1c, d2c)

    @staticmethod
    def backward(ctx, grad_kld):
        d1, d2 = ctx.saved_tensors
        g = grad_kld.detach().to(torch.float32).contiguous()
        g1, g2 = torch.empty_like(d1), torch.empty_like(d2)
        n, c, h, w = d1.shape
        with torch.cuda.device(d1.device):
            st = _lib.load().mspl_kld_bwd(_ptr(d1), _ptr(d2), _ptr(g), n, c, h * w, _ptr(g1), _ptr(g2), _stream(d1.device))
        _lib.check(st, "mspl_kld_bwd")
        return g1, g2


def pixelwise_kld(d1, d2):
    """PixelwiseKLD.forward (loss_fns/segmentation_loss.py:181-189), differentiable w.r.t. both inputs."""
    _require_cuda(d1, "dist1", torch.float32, 4)
    _require_cuda(d2, "dist2", torch.float32, 4)
    if d1.shape != d2.shape:
        raise ValueError("dist1/dist2 shapes differ")
    return _PixelwiseKLD.apply(d1, d2)


class _UwLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, u, cw, norm_pixels):
        pred_c, u_c = pred.detach().contiguous(), u.detach().contiguous()
        n, k, h, w = pred_c.shape
        dev = pred_c.device
        loss = torch.empty((), dtype=torch.float32, device=dev)
        ws = _workspace(dev)
        norm = float(norm_pixels) if norm_pixels is not None else float(n * h * w)
        with torch.cuda.device(dev):
            st = _lib.load().mspl_uw_loss_fwd(_ptr(pred_c), _ptr(target), _ptr(u_c), _ptr(cw), n, k, h * w, norm, _ptr(loss),
                                              _ptr(ws), ws.numel(), _stream(dev))
        _lib.check(st, "mspl_uw_loss_fwd")
        ctx.save_for_backward(pred_c, target, u_c, cw)
        ctx.norm = norm
        ctx.u_shape = u.shape
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        pred, target, u, cw = ctx.saved_tensors
        n, k, h, w = pred.shape
        g = grad_loss.detach().to(torch.float32).reshape(1).contiguous()
        d_pred = torch.empty_like(pred)
        d_u = torch.empty_like(u) if ctx.needs_input_grad[2] else None
        with torch.cuda.device(pred.device):
            st = _lib.load().mspl_uw_loss_bwd(_ptr(pred), _ptr(target), _ptr(u), _ptr(cw), _ptr(g), n, k, h * w, ctx.norm,
                                              _ptr(d_pred), _ptr(d_u), _stream(pred.device))
        _lib.check(st, "mspl_uw_loss_bwd")
        return d_pred, None, (d_u.reshape(ctx.u_shape) if d_u is not None else None), None, None


def uw_segmentation_loss(pred, target, u_weight, class_weights, norm_pixels=None):
    """UncertaintyWeightedSegmentationLoss.forward (loss_fns/segmentation_loss.py:155-175): mean over ALL pixels of
    w[t] * (-log_softmax(pred)[t]) * exp(-u); differentiable w.r.t. pred and u_weight."""
    _require_cuda(pred, "pred", torch.float32, 4)
    n, k, h, w = pred.shape
    target = _require_cuda(target, "target", torch.int64)
    if target.numel() != n * h * w:
        raise ValueError("target must hold one class index per pixel")
    if not u_weight.is_cuda or u_weight.dtype != torch.float32 or u_weight.numel() != n * h * w:
        raise ValueError("u_weight must be a CUDA fp32 tensor with one value per pixel")
    cw = _require_cuda(class_weights, "class_weights", torch.float32, 1)
    if cw.numel() != k:
        raise ValueError("class_weights must have %d entries" % k)
    return _UwLoss.apply(pred, target, u_weight, cw, norm_pixels)


def miou_counts(output, target, num_classes, counts=None):
    """GPU MIOU.get_iou counting (utilities/metrics/segmentation_miou.py:13-44).  output: (B,C,H,W) fp32 logits (argmax over
    classes is taken, first maximal index) or a (B,H,W) uint8/int64 label map; target: integer label map (255 = dropped).
    Returns an int64 (3, num_classes) tensor [area_inter, area_pred, area_mask] (accumulated into `counts` if given)."""
    if not isinstance(output, torch.Tensor) or not output.is_cuda:
        raise ValueError("output must be a CUDA tensor (mspl_b200 has no CPU path)")
    dev = output.device
    target = target.to(device=dev, dtype=torch.int64).contiguous()
    if counts is None:
        counts = torch.zeros((3, num_classes), dtype=torch.int64, device=dev)
    _require_cuda(counts, "counts", torch.int64)
    lib = _lib.load()
    with torch.cuda.device(dev):
        if output.dim() == 4:
            out = _require_cuda(output.detach().float().contiguous(), "output", torch.float32, 4)
            n, c, h, w = out.shape
            if target.numel() != n * h * w:
                raise ValueError("target must hold one label per pixel")
            st = lib.mspl_miou_from_logits(_ptr(out), _ptr(target), n, c, h * w, num_classes, _ptr(counts), _stream(dev))
        else:
            pred = output.detach().contiguous()
            if pred.dtype not in (torch.uint8, torch.int64):
                pred = pred.to(torch.int64)
            if target.numel() != pred.numel():
                raise ValueError("pred/target sizes differ")
            st = lib.mspl_miou_from_labels(_ptr(pred), int(pred.dtype == torch.int64), _ptr(target), pred.numel(), num_classes,
                                           _ptr(counts), _stream(dev))
    _lib.check(st, "mspl_miou")
    return counts


# ---- NIDLoss ------------------------------------------------------------------------------------------------------------
_nid_workspaces = {}


class _NidLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, camera, label, image_bins, label_bins, bw_camera, bw_label):
        cam = _require_cuda(camera.detach().float().contiguous(), "camera", torch.float32, 4)
        lab = _require_cuda(label.detach().float().contiguous(), "label", torch.float32, 4)
        b, three, h, w = cam.shape
        if three != 3 or lab.shape[0] != b or lab.shape[2:] != (h, w):
            raise ValueError("camera must be (B,3,H,W) and label (B,C,H,W) with the same B, H, W")
        dev = cam.device
        lib = _lib.load()
        key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
        ws = _nid_workspaces.get(key)
        if ws is None:
            ws = _nid_workspaces[key] = torch.zeros(lib.mspl_nid_workspace_bytes(), dtype=torch.uint8, device=dev)
        state = torch.empty(lib.mspl_nid_state_bytes() // 4, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            st = lib.mspl_nid_fwd(_ptr(cam), _ptr(lab), b, lab.shape[1], h * w, int(image_bins), int(label_bins), float(bw_camera),
                                  float(bw_label), _ptr(ws), ws.numel(), _ptr(state), _stream(dev))
        _lib.check(st, "mspl_nid_fwd")
        ctx.save_for_backward(cam, lab, state)
        ctx.cfg = (int(image_bins), int(label_bins), float(bw_camera), float(bw_label))
        return state[0].clone()

    @staticmethod
    def backward(ctx, grad_loss):
        cam, lab, state = ctx.saved_tensors
        k, lb, bwc, bwl = ctx.cfg
        b, c, h, w = lab.shape
        g = grad_loss.detach().to(torch.float32).reshape(1).contiguous()
        d_label = torch.empty_like(lab)
        with torch.cuda.device(lab.device):
            st = _lib.load().mspl_nid_bwd(_ptr(cam), _ptr(lab), _ptr(g), b, c, h * w, k, lb, bwc, bwl, _ptr(state), _ptr(d_label),
                                          _stream(lab.device))
        _lib.check(st, "mspl_nid_bwd")
        return None, d_label, None, None, None, None


def nid_loss(camera, label, image_bins=16, label_bins=4, bw_camera=0.005, bw_label=0.001):
    """NIDLoss.forward (loss_fns/segmentation_loss.py:101-118): (NID(grey(camera), soft-argmax(label)) - 0.95) * 20,
    differentiable w.r.t. the label logits."""
    if image_bins > 32 or label_bins > 8:
        raise NotImplementedError("nid_loss supports up to 32 image bins and 8 label bins")
    return _NidLoss.apply(camera, label, image_bins, label_bins, bw_camera, bw_label)


# ---- in-training visualisation maps -------------------------------------------------------------------------------------
def prediction_maps(main, aux=None, want_heat=True):
    """Device half of in_training_visualization_img (utilities/utils.py:76-133): returns (predictions int64 (N,H,W) =
    first-argmax of ``main + 0.5*aux`` (of ``main`` when aux is None), heat f32 (N,1,H,W) = ``-kld / max(kld) + 1`` with
    ``kld = PixelwiseKLD(main, aux)``, or None without aux / with want_heat=False).  Two launches, no host sync."""
    main = _require_cuda(main.detach().float().contiguous(), "main", torch.float32, 4)
    if aux is not None:
        aux = _require_cuda(aux.detach().float().contiguous(), "aux", torch.float32, 4)
        if aux.shape != main.shape:
            raise ValueError("main/aux shapes differ")
    n, c, h, w = main.shape
    dev = main.device
    labels = torch.empty((n, h, w), dtype=torch.int64, device=dev)
    heat_wanted = want_heat and aux is not None
    kld = torch.empty((n, h, w), dtype=torch.float32, device=dev) if heat_wanted else None
    key = torch.zeros(1, dtype=torch.int32, device=dev) if heat_wanted else None
    lib = _lib.load()
    with torch.cuda.device(dev):
        st = _stream(dev)
        _lib.check(lib.mspl_prediction_maps(_ptr(main), _ptr(aux), n, c, h * w, _ptr(labels), _ptr(kld), _ptr(key), st),
                   "mspl_prediction_maps")
        heat = None
        if heat_wanted:
            heat = torch.empty((n, 1, h, w), dtype=torch.float32, device=dev)
            _lib.check(lib.mspl_kld_heatmap(_ptr(kld), kld.numel(), _ptr(key), _ptr(heat), st), "mspl_kld_heatmap")
    return labels, heat


def label_colors(labels, colors):
    """LongTensorToRGBPIL (utilities/utils.py:188-237) for a batch on the device: labels (N,H,W) integer CUDA tensor, colors a
    sequence of (r, g, b) triples indexed by class id -> uint8 (N,3,H,W).  Labels outside the table give black."""
    if not isinstance(labels, torch.Tensor) or not labels.is_cuda:
        raise ValueError("labels must be a CUDA tensor (mspl_b200 has no CPU path)")
    if labels.dim() != 3:
        raise ValueError("labels must be (N,H,W)")
    labels = labels.to(torch.int64).contiguous()
    table = [int(v) for rgb in colors for v in rgb]
    if len(table) % 3 or len(table) > 3 * 256 or any(v < 0 or v > 255 for v in table):
        raise ValueError("colors must be at most 256 (r, g, b) triples of bytes")
    n, h, w = labels.shape
    rgb = torch.empty((n, 3, h, w), dtype=torch.uint8, device=labels.device)
    buf = (ctypes.c_ubyte * max(1, len(table)))(*table)
    with torch.cuda.device(labels.device):
        st = _lib.load().mspl_label_colors(_ptr(labels), n, h * w, buf, len(table) // 3, _ptr(rgb), _stream(labels.device))
    _lib.check(st, "mspl_label_colors")
    return rgb
