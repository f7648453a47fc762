"""CPU: argument checks of mspl_uw_ce_step_half, the fp16 / bf16 entry of K4.  The device pointers are fake, so every call
below has to return before any CUDA work (a call that got as far as a launch would report a CUDA error)."""
import os

import pytest

BAD, ALIGN = -1, -2
F16, BF16 = 1, 2


@pytest.fixture(scope="module")
def lib():
    from mspl_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


def _status(lib, dtype=BF16, k=5, odd_logits=False, d_aux=True, u8=True):
    fake = 1 << 32
    main, aux, target, cw, out3, d_main, d_aux_p, ws = (fake + (i << 28) for i in range(8))
    if odd_logits:
        main += 1
    return lib.mspl_uw_ce_step_half(main, aux, dtype, target, int(u8), cw, 1, k, 256 * 480, 20.0, 256.0 * 480, 1.0, None, out3,
                                    d_main, d_aux_p if d_aux else None, None, ws, lib.mspl_uw_ce_workspace_bytes(), None)


def test_half_entry_rejects_bad_arguments(lib):
    for kw, want in ((dict(dtype=0), BAD), (dict(dtype=3), BAD), (dict(d_aux=False), BAD), (dict(k=0), BAD),
                     (dict(odd_logits=True), ALIGN), (dict(odd_logits=True, dtype=F16, u8=False), ALIGN)):
        assert _status(lib, **kw) == want, kw
