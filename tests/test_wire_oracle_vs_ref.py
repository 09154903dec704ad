"""oracle/wire_oracle.py's restatement of the live driver's phosphor decay against the reference's own function: the lines
of fade_phosphors() are cut out of the reference's crt_main.c (437-452; that branch of the file needs an external windowing
library and cannot be compiled whole) into a scratch translation unit by oracle/Makefile (libref_fade.so).  This is what
pins `crtx_fade_phosphors` (tests/test_gpu_wire.py) to the reference rather than to our own reading of it."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import support as S

sys.path.insert(0, S.ORACLE_DIR)
import wire_oracle as W  # noqa: E402

REF = os.path.join(S.REF_DIR, "libref_fade.so")


@pytest.mark.parametrize("w,h,seed", [(832, 624, 1), (53, 37, 2), (1, 1, 3), (640, 480, 4)])
def test_fade_phosphors_restatement_is_the_reference_function(w, h, seed):
    """(where libref_fade.so is not built, against the reference's images recorded under tests/golden/reference/)"""
    live = os.path.exists(REF)
    R = C.CDLL(REF) if live else None
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 1 << 32, size=w * h, dtype=np.uint32)
    img[:4] = (0, 0xFFFFFFFF, 0x00FFFFFF, 0xFF000000)[: min(4, img.size)]
    ours = img.copy()
    theirs = img.astype(np.int32).copy()

    def ref_step():
        R.ref_fade_phosphors(theirs.ctypes.data_as(C.c_void_p), w, h)
        return S.digest(theirs.view(np.uint32))
    for _ in range(6):  # the live loop applies it frame after frame
        ours = W.fade_phosphors(ours).astype(np.uint32)
        assert S.digest(ours) == S.ref_result(ref_step, live)
        if live:
            assert np.array_equal(ours, theirs.view(np.uint32))
