"""ctypes binding of libmspl_b200.so (the C ABI in include/mspl_b200.h).

There is deliberately no fallback: if the shared library is missing the import of any op raises, and every
op refuses tensors that are not on a CUDA device.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MSPL_B200_LIB", os.path.join(_HERE, "lib", "libmspl_b200.so"))

c_i64, c_int, c_f32, c_f64, c_vp, c_sz = (ctypes.c_int64, ctypes.c_int, ctypes.c_float, ctypes.c_double,
                                          ctypes.c_void_p, ctypes.c_size_t)

# name -> (restype, argtypes); must list every symbol include/mspl_b200.h declares (tests check this)
SIGNATURES = {
    "mspl_strerror": (ctypes.c_char_p, [c_int]),
    "mspl_abi_version": (c_int, []),
    "mspl_fuse_variant": (ctypes.c_char_p, []),
    "mspl_softmax_kld": (c_int, [c_vp, c_vp, c_i64, c_int, c_i64, c_vp, c_vp, c_vp]),
    "mspl_fuse_sources": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_int, c_int, c_int, c_int, c_int,
                                  c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mspl_fuse_sources_lowres": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_int, c_int, c_int,
                                         c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mspl_class_order": (c_int, [c_vp, c_int, c_int, c_vp, c_vp, c_vp]),
    "mspl_class_order_votes": (c_int, [c_vp, c_int, c_int, c_vp, c_vp]),
    "mspl_class_order_shape": (c_int, [c_vp, c_int, c_int]),
    "mspl_vote_labels": (c_int, [c_vp, c_int, c_i64, c_int, c_int, c_int, c_vp, c_vp]),
    "mspl_radix_state_bytes": (c_sz, [c_int]),
    "mspl_conf_hist": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_int, c_vp]),
    "mspl_bracket_select": (c_int, [c_vp, c_int, c_f64, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mspl_bracket_classify": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mspl_cand_hist_pass": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_int, c_vp]),
    "mspl_cand_select": (c_int, [c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_int, c_vp]),
    "mspl_cand_resolve": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mspl_cand_apply": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_vp]),
    "mspl_radix_hist_pass": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_int, c_vp, c_vp, c_int, c_vp]),
    "mspl_radix_select": (c_int, [c_vp, c_int, c_int, c_f64, c_vp, c_vp, c_vp, c_vp]),
    "mspl_apply_thresholds": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_vp]),
    "mspl_uw_ce_workspace_bytes": (c_sz, []),
    "mspl_uw_ce_fwd_bwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_i64, c_f32, c_f64, c_f32, c_vp, c_vp,
                                   c_vp, c_vp, c_sz, c_vp]),
    "mspl_uw_ce_fwd_bwd_u8": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_i64, c_f32, c_f64, c_f32, c_vp, c_vp,
                                      c_vp, c_vp, c_sz, c_vp]),
    "mspl_uw_ce_step": (c_int, [c_vp, c_vp, c_vp, c_int, c_vp, c_i64, c_int, c_i64, c_f32, c_f64, c_f32, c_vp, c_vp, c_vp, c_vp,
                                c_vp, c_sz, c_vp]),
    "mspl_uw_ce_lowres_fwd_bwd_u8": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_f32,
                                             c_f64, c_f32, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "mspl_uw_ce_lowres_fwd_bwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_f32, c_f64,
                                          c_f32, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "mspl_scale_inplace": (c_int, [c_vp, c_i64, c_vp, c_vp]),
    "mspl_kld_fwd": (c_int, [c_vp, c_vp, c_i64, c_int, c_i64, c_vp, c_vp]),
    "mspl_kld_bwd": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_i64, c_vp, c_vp, c_vp]),
    "mspl_uw_loss_fwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_i64, c_f64, c_vp, c_vp, c_sz, c_vp]),
    "mspl_uw_loss_bwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_i64, c_f64, c_vp, c_vp, c_vp]),
    "mspl_nid_workspace_bytes": (c_sz, []),
    "mspl_nid_state_bytes": (c_sz, []),
    "mspl_nid_fwd": (c_int, [c_vp, c_vp, c_i64, c_int, c_i64, c_int, c_int, c_f32, c_f32, c_vp, c_sz, c_vp, c_vp]),
    "mspl_nid_bwd": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_i64, c_int, c_int, c_f32, c_f32, c_vp, c_vp, c_vp]),
    "mspl_prediction_maps": (c_int, [c_vp, c_vp, c_i64, c_int, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mspl_kld_heatmap": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp]),
    "mspl_label_colors": (c_int, [c_vp, c_i64, c_i64, c_vp, c_int, c_vp, c_vp]),
    "mspl_miou_from_logits": (c_int, [c_vp, c_vp, c_i64, c_int, c_i64, c_int, c_vp, c_vp]),
    "mspl_miou_from_labels": (c_int, [c_vp, c_int, c_vp, c_i64, c_int, c_vp, c_vp]),
}

_lib = None


class MsplError(RuntimeError):
    pass


def load():
    """Load (once) and return the ctypes handle; raises MsplError if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise MsplError("libmspl_b200.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; "
                        "g.build()'` or `make -C mspl_b200/csrc`; there is no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def check(status, what):
    if status != 0:
        raise MsplError("%s failed: %s (%d)" % (what, load().mspl_strerror(status).decode(), status))
