"""CPU: the C-ABI library loads and exports exactly the symbols include/mspl_b200.h declares; the product package
never touches the oracle."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "mspl_b200.h")).read()
    return sorted(set(re.findall(r"^MSPL_API\s+[\w\s\*]+?\b(mspl_\w+)\s*\(", text, flags=re.M)))


@pytest.fixture(scope="module")
def lib():
    from mspl_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


def test_header_declares_entry_points():
    names = _declared()
    assert len(names) >= 17 and "mspl_fuse_sources" in names and "mspl_uw_ce_fwd_bwd" in names


def test_library_exports_every_declared_symbol(lib):
    from mspl_b200 import _lib
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.LIB_PATH], text=True)
    exported = set(re.findall(r"\sT\s+(mspl_\w+)", out))
    assert set(_declared()) <= exported, sorted(set(_declared()) - exported)
    assert exported == set(_declared()), "exported but undeclared: %s" % sorted(exported - set(_declared()))
    assert set(_lib.SIGNATURES) == set(_declared())
    for name in _declared():
        assert getattr(lib, name) is not None


def test_host_only_entry_points(lib):
    assert lib.mspl_abi_version() == 5
    assert lib.mspl_strerror(0) == b"ok" and b"misaligned" in lib.mspl_strerror(-2)
    assert lib.mspl_radix_state_bytes(5) == 5 * 32
    assert lib.mspl_uw_ce_workspace_bytes() >= 16 + 2 * 8 * 148
    assert b"CH=" in lib.mspl_fuse_variant()


def test_sass_is_sm100a():
    from mspl_b200 import _lib
    out = subprocess.check_output(["cuobjdump", "-lelf", _lib.LIB_PATH], text=True)
    assert "sm_100a" in out and "sm_90" not in out


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "mspl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), os.path.join(dirpath, f)
                assert "mspl_oracle" not in text, os.path.join(dirpath, f)


def test_ops_refuse_cpu_tensors():
    import torch
    from mspl_b200 import ops
    with pytest.raises(ValueError, match="CUDA"):
        ops.softmax_kld(torch.zeros(1, 3, 4, 4), torch.zeros(1, 3, 4, 4))
    with pytest.raises(ValueError, match="CUDA"):
        ops.pixelwise_kld(torch.zeros(1, 3, 4, 4), torch.zeros(1, 3, 4, 4))
    assert ops.vote_threshold(3, None) == 2 and ops.vote_threshold(3, 'all') == 3 and ops.vote_threshold(3, 1) == 1
    assert ops.vote_threshold(3, 7) == 2 and ops.vote_threshold(3, '3') == 2 and ops.vote_threshold(2, 'half') == 2


def test_header_is_plain_c_and_links_from_c(lib, tmp_path):
    """The boundary is a C ABI: the header compiles as C99 and a C program links against the library and calls its host-only
    entry points (what a cgo / JNI / ctypes-free binding would do)."""
    from mspl_b200 import _lib
    src = tmp_path / "abi_smoke.c"
    src.write_text('#include <stdio.h>\n#include <string.h>\n#include "mspl_b200.h"\n'
                   'int main(void) {\n'
                   '    if (mspl_abi_version() != MSPL_ABI_VERSION) return 1;\n'
                   '    if (strcmp(mspl_strerror(MSPL_OK), "ok") != 0) return 2;\n'
                   '    if (mspl_radix_state_bytes(MSPL_MAX_CLASSES) == 0 || mspl_uw_ce_workspace_bytes() == 0) return 3;\n'
                   '    /* argument validation happens before any CUDA call: usable without a device */\n'
                   '    if (mspl_fuse_sources(0, NULL, NULL, NULL, NULL, 0, 0, 5, 0, 2, 4, 1, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL)\n'
                   '        != MSPL_ERR_BAD_ARG) return 4;\n'
                   '    printf("%s\\n", mspl_fuse_variant());\n'
                   '    return 0;\n}\n')
    exe = tmp_path / "abi_smoke"
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-L", libdir,
                           "-lmspl_b200", "-Wl,-rpath," + libdir, "-o", str(exe)])
    out = subprocess.check_output([str(exe)], text=True)
    assert "CH=" in out


def test_class_order_groups_classes_by_target(lib):
    """Host logic of K1's grouped class order (no GPU): a permutation of the classes sorted by (target, class index), one
    boundary bit per target group, the `present` mask -- for the reference's three tables and for awkward ones."""
    import ctypes
    import numpy as np
    from mspl_b200.data_loader.segmentation.greenhouse import SOURCE_TABLES
    tables = [np.asarray(t) for t in SOURCE_TABLES.values()]
    tables += [np.array([2]), np.array([3, 0, 1, 0, 3, 1, 2, 2, 0, 1, 3]), np.arange(256) % 5, np.array([1] * 7)]
    for lut in tables:
        C = len(lut)
        buf = (ctypes.c_ubyte * C)(*[int(v) for v in lut])
        row = (ctypes.c_ubyte * C)()
        seg = (ctypes.c_ubyte * 64)()
        present = ctypes.c_uint32(0)
        ch = lib.mspl_class_order(buf, C, 5, row, seg, ctypes.byref(present))
        assert ch >= 4
        order = np.array(list(row))
        assert sorted(order.tolist()) == list(range(C))                                  # a permutation
        tgt = lut[order]
        assert np.array_equal(order, np.array(sorted(range(C), key=lambda c: (lut[c], c))))  # by (target, class index)
        bits = [(seg[i // ch] >> (i % ch)) & 1 for i in range(C)]
        want = [int(i == C - 1 or tgt[i + 1] != tgt[i]) for i in range(C)]
        assert bits == want                                                               # one boundary per target group
        assert present.value == sum(1 << int(k) for k in set(lut.tolist()))
        assert sum(bits) == bin(present.value).count("1")
        # the epilogue's companion table: one vote increment per target group in visiting (= ascending target) order
        vote = (ctypes.c_uint32 * 8)()
        nchunk = ctypes.c_uint32(0)
        ngroup = lib.mspl_class_order_votes(buf, C, 5, vote, ctypes.byref(nchunk))
        targets = sorted(set(int(k) for k in lut.tolist()))
        assert ngroup == len(targets) and nchunk.value == -(-C // ch)
        assert list(vote)[:ngroup] == [1 << (4 * k) for k in targets] and not any(list(vote)[ngroup:])
    bad = (ctypes.c_ubyte * 3)(1, 2, 7)
    assert lib.mspl_class_order(bad, 3, 5, (ctypes.c_ubyte * 3)(), (ctypes.c_ubyte * 64)(), ctypes.byref(ctypes.c_uint32())) == -1
    assert lib.mspl_class_order_votes(bad, 3, 5, (ctypes.c_uint32 * 8)(), ctypes.byref(ctypes.c_uint32())) == -1


def _fuse_status(lib, lowres, S=3, C=13, K=5, policy=0, ignore=4, ds_rate=1, conf=True, conf_hist=True, bad_entry=False,
                 misaligned=False, head=(64, 120), out=(256, 480)):
    """Status of one K1 entry point call whose device pointers are fake: the argument checks only test their alignment, so
    every call below has to return before any CUDA work (a call that got as far as a launch would report a CUDA error)."""
    import ctypes
    vp, n = ctypes.c_void_p, 9
    fake = 1 << 32
    main = (vp * n)(*[fake + (s << 24) + (2 if misaligned and s == 0 else 0) for s in range(n)])
    aux = (vp * n)(*[fake + ((n + s) << 24) for s in range(n)])
    ncls = (ctypes.c_int * n)(*[C] * n)
    tables = [(ctypes.c_ubyte * 256)(*[c % 5 for c in range(256)]) for _ in range(n)]
    if bad_entry:
        tables[1][2] = K
    lut = (vp * n)(*[ctypes.addressof(t) for t in tables])
    label, conf_p, unc, class_hist, hist = (fake + (i << 28) for i in range(1, 6))
    common = [K, policy, 2, ignore, ds_rate, label, conf_p if conf else None, unc, None, class_hist,
              hist if conf_hist else None, None, None]
    if lowres:
        main_hw = (ctypes.c_int * (2 * n))(*[2 * v for v in head] * n)
        aux_hw = (ctypes.c_int * (2 * n))(*list(head) * n)
        return lib.mspl_fuse_sources_lowres(S, main, aux, ncls, lut, main_hw, aux_hw, 1, out[0], out[1], *common)
    return lib.mspl_fuse_sources(S, main, aux, ncls, lut, 1, out[0] * out[1], *common)


@pytest.mark.parametrize("lowres", [False, True])
def test_fuse_entry_points_reject_bad_arguments(lib, lowres):
    """Argument checks of mspl_fuse_sources and mspl_fuse_sources_lowres, one invalid argument per call (no GPU).  One image
    throughout: a call without images returns MSPL_OK before the per-source checks."""
    BAD, ALIGN, UNSUPPORTED = -1, -2, -3
    cases = [(dict(S=0), BAD), (dict(S=9), BAD), (dict(K=1), BAD), (dict(K=9), BAD), (dict(policy=2), BAD),
             (dict(ignore=5), BAD), (dict(conf=False), BAD), (dict(C=0), BAD), (dict(C=257), BAD),
             (dict(bad_entry=True), BAD), (dict(ds_rate=0), BAD), (dict(misaligned=True), ALIGN)]
    if lowres:
        cases += [(dict(head=(0, 120)), BAD), (dict(head=(64, 0)), BAD), (dict(out=(3, 5)), UNSUPPORTED)]
    for kw, want in cases:
        assert _fuse_status(lib, lowres, **kw) == want, kw


def test_vote_threshold_follows_merge_outputs_rule():
    """merge_outputs' threshold rule (uest_seg_multi_os.py:697-705): None / 'half' / anything else -> S//2+1, 'all' -> S, an int
    (bool included, as `isinstance(thresh, int)` accepts it) <= S -> itself."""
    from mspl_b200.ops import vote_threshold
    assert vote_threshold(3, None) == 2 and vote_threshold(3, 'half') == 2 and vote_threshold(3, 'all') == 3
    assert vote_threshold(3, 1) == 1 and vote_threshold(3, 3) == 3 and vote_threshold(3, 4) == 2
    assert vote_threshold(3, True) == 1 and vote_threshold(3, False) == 0
    assert vote_threshold(3, '2') == 2 and vote_threshold(4, 'nonsense') == 3 and vote_threshold(1, None) == 1
    # the oracle's restatement follows the same rule, bool included
    from oracle import mspl_oracle as O
    for S in (1, 2, 3, 4, 8, 15):
        for t in [None, 'half', 'all', '3', 'nonsense', True, False] + list(range(-1, S + 3)):
            assert O.vote_threshold(S, t) == vote_threshold(S, t), (S, t)
