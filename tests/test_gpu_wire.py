"""SURVEY 8f-2 / 8f-4: the image wire formats on the device (BMP and PPM pixel data <-> the loaders' int pixels) and
the live driver's phosphor decay, against numpy restatements of bmp_rw.c / ppm_rw.c / crt_main.c:437-452
(oracle/wire_oracle.py).  Byte shuffles: bit-exact, including sizes that are not multiples of the vector widths."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import support as S

sys.path.insert(0, os.path.join(S.ROOT, "oracle"))
import wire_oracle as W  # noqa: E402

pytestmark = pytest.mark.gpu


def lib():
    from ntsc_crt_b200 import capi
    L = capi.load("ntsc")
    vp, ip = C.c_void_p, C.c_int
    L.crtx_bmp_unpack.argtypes = [vp, vp, ip, ip, ip, vp]
    L.crtx_bmp_pack.argtypes = [vp, vp, ip, ip, vp]
    L.crtx_ppm_unpack.argtypes = [vp, vp, ip, ip, ip, vp]
    L.crtx_ppm_pack.argtypes = [vp, vp, ip, ip, vp]
    L.crtx_fade_phosphors.argtypes = [vp, C.c_size_t, vp]
    L.crtx_last_error.restype = C.c_char_p
    return L


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def host(t, dtype, count):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy().view(dtype)[:count]


@pytest.mark.parametrize("w,h,bits", [(640, 480, 32), (321, 7, 24), (2, 3, 24), (833, 5, 32), (1, 1, 24)])
def test_bmp_wire_format(w, h, bits):
    import torch
    L = lib()
    rng = np.random.default_rng(w * h + bits)
    rowbytes = (w * (bits // 8) + 3) & ~3
    filebytes = rng.integers(0, 256, size=rowbytes * h, dtype=np.uint8)
    d_file, d_img = dev(filebytes), torch.zeros(w * h * 4, dtype=torch.uint8, device="cuda")
    assert L.crtx_bmp_unpack(d_img.data_ptr(), d_file.data_ptr(), w, h, bits, None) == 0, L.crtx_last_error()
    want = W.bmp_unpack(filebytes.tobytes(), w, h, bits)
    got = host(d_img, np.uint32, w * h).reshape(h, w)
    assert np.array_equal(got, want)
    d_back = torch.zeros(w * h * 4, dtype=torch.uint8, device="cuda")
    assert L.crtx_bmp_pack(d_back.data_ptr(), d_img.data_ptr(), w, h, None) == 0, L.crtx_last_error()
    assert np.array_equal(host(d_back, np.uint32, w * h).reshape(h, w), W.bmp_pack(want, w, h))


@pytest.mark.parametrize("w,h,maxc,skew", [(832, 624, 255, 0), (333, 7, 255, 0), (5, 3, 100, 0), (2, 1, 1, 0), (97, 13, 255, 1),
                                           (64, 3, 31, 3)])
def test_ppm_wire_format(w, h, maxc, skew):
    """skew: byte offset of the file's pixel data inside its buffer (after a header the data is rarely word aligned)"""
    import torch
    L = lib()
    rng = np.random.default_rng(w * 7 + h + maxc)
    filebytes = rng.integers(0, maxc + 1, size=3 * w * h, dtype=np.uint8)
    buf = np.zeros(3 * w * h + 16, dtype=np.uint8)
    buf[skew:skew + 3 * w * h] = filebytes
    d_buf, d_img = dev(buf), torch.zeros(w * h * 4, dtype=torch.uint8, device="cuda")
    assert L.crtx_ppm_unpack(d_img.data_ptr(), d_buf.data_ptr() + skew, w, h, maxc, None) == 0, L.crtx_last_error()
    want = W.ppm_unpack(filebytes.tobytes(), w, h, maxc)
    assert np.array_equal(host(d_img, np.uint32, w * h).reshape(h, w), want)
    # pack: any int pixels (the decoder's output carries alpha 0xff in the top byte; ppm_rw.c drops it)
    img = rng.integers(0, 1 << 32, size=w * h, dtype=np.uint32)
    d_src, d_out = dev(img), torch.full((3 * w * h + 16,), 0xEE, dtype=torch.uint8, device="cuda")
    assert L.crtx_ppm_pack(d_out.data_ptr() + skew, d_src.data_ptr(), w, h, None) == 0, L.crtx_last_error()
    got = host(d_out, np.uint8, 3 * w * h + 16)
    assert np.array_equal(got[skew:skew + 3 * w * h], W.ppm_pack(img, w, h))
    assert np.all(got[:skew] == 0xEE) and np.all(got[skew + 3 * w * h:] == 0xEE), "wrote outside the pixel data"
    assert L.crtx_ppm_unpack(d_img.data_ptr(), d_buf.data_ptr(), w, h, 256, None) != 0  # ppm_rw.c:57-62 rejects it too


@pytest.mark.parametrize("npix,skew", [(832 * 624, 0), (1003, 0), (3, 0), (4097, 1), (1, 3)])
def test_fade_phosphors(npix, skew):
    """skew: pixels between a 16-byte boundary and the image start (the scalar path)"""
    import torch
    L = lib()
    rng = np.random.default_rng(npix)
    img = rng.integers(0, 1 << 32, size=npix + 8, dtype=np.uint32)
    d = dev(img)
    assert L.crtx_fade_phosphors(d.data_ptr() + 4 * skew, npix, None) == 0, L.crtx_last_error()
    got = host(d, np.uint32, npix + 8)
    want = img.copy()
    want[skew:skew + npix] = W.fade_phosphors(img[skew:skew + npix])
    assert np.array_equal(got, want)
    for _ in range(3):  # repeated decay, as the live loop applies it frame after frame
        assert L.crtx_fade_phosphors(d.data_ptr() + 4 * skew, npix, None) == 0
        want[skew:skew + npix] = W.fade_phosphors(want[skew:skew + npix])
    assert np.array_equal(host(d, np.uint32, npix + 8), want)
    # ... and against the reference's own function, cut out of crt_main.c:437-452 and compiled (oracle/Makefile: libref_fade.so)
    import ctypes as C
    import os
    # (where it is not built: the reference's image recorded under tests/golden/reference/)
    ref = os.path.join(S.REF_DIR, "libref_fade.so")

    def ref_fade():
        R = C.CDLL(ref)
        theirs = img[skew:skew + npix].astype(np.int32).copy()
        for _ in range(4):
            R.ref_fade_phosphors(theirs.ctypes.data_as(C.c_void_p), npix, 1)
        return S.digest(theirs.view(np.uint32))
    assert S.digest(host(d, np.uint32, npix + 8)[skew:skew + npix]) == S.ref_result(ref_fade, os.path.exists(ref))
