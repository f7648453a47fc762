"""CPU: K1's compiled chunk shapes (kSourceShapes, pixel_math.cuh) are exactly the class orders build_class_order produces for
the greenhouse tables, so each shipped source runs its straight-line body; every other table runs the generic chunk loop."""
import ctypes
import os

import numpy as np
import pytest

from mspl_b200.data_loader.segmentation.greenhouse import SOURCE_TABLES


@pytest.fixture(scope="module")
def lib():
    from mspl_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


def _shape(lib, lut, K=5):
    lut = np.asarray(lut)
    return lib.mspl_class_order_shape((ctypes.c_ubyte * len(lut))(*[int(v) for v in lut]), len(lut), K)


def _order(lib, lut):
    C = len(lut)
    row, seg, present = (ctypes.c_ubyte * C)(), (ctypes.c_ubyte * 64)(), ctypes.c_uint32(0)
    ch = lib.mspl_class_order((ctypes.c_ubyte * C)(*[int(v) for v in lut]), C, 5, row, seg, ctypes.byref(present))
    return ch, list(seg)[:-(-C // ch)]


def test_shipped_tables_have_compiled_shapes(lib):
    """A shape matches only when (C, nchunk, seg) equal the listed entry, so three distinct non-zero ids for the three shipped
    tables mean the list holds exactly their orders.  The ids do not depend on the number of target classes."""
    ids = {name: _shape(lib, lut) for name, lut in SOURCE_TABLES.items()}
    assert sorted(ids.values()) == [1, 2, 3], ids
    assert ids == {name: _shape(lib, lut, K=8) for name, lut in SOURCE_TABLES.items()}
    # the listed words, as the kernel's bodies use them (bit j of chunk i: slot j ends its target group)
    want = {"camvid": [0x01, 0x0a, 0x04], "cityscapes": [0x01, 0x00, 0x04, 0x11], "forest": [0x1a]}
    for name, lut in SOURCE_TABLES.items():
        ch, seg = _order(lib, lut)
        assert ch == 5 and seg == want[name], (name, seg)


def test_other_tables_run_the_chunk_loop(lib):
    """Tables with the shipped class counts but other groupings, and other class counts, get shape 0."""
    gen = np.random.default_rng(7)
    cam = np.asarray(SOURCE_TABLES["camvid"])
    others = [cam[::-1], np.roll(SOURCE_TABLES["cityscapes"], 1), np.array([1, 1, 2, 2, 3]), np.array([2] * 13),
              np.arange(256) % 5, np.array([3]), np.append(cam, 1)]
    others += [gen.integers(0, 5, size=c) for c in (13, 20, 5) for _ in range(20)]
    shipped = {tuple(_order(lib, lut)[1]) + (len(lut),) for lut in SOURCE_TABLES.values()}
    for lut in others:
        same_order = tuple(_order(lib, lut)[1]) + (len(lut),) in shipped
        assert (_shape(lib, lut) != 0) == same_order, lut
    assert _shape(lib, np.array([1, 2, 7]), K=5) == -1
