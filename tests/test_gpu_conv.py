"""GPU parity of the USE_CONVOLUTION decoder variant (SURVEY 8a row a11: crt_core.c:85-147, the 7-tap FIR
eqf): libcrt_b200_ntsc_conv.so against the oracle's FIR line pass and the reference compiled with USE_CONVOLUTION 1
(oracle/_ref, else its states recorded under tests/golden/reference/) -- bit for bit, through the drop-in C-ABI and the
batch one."""
import numpy as np
import pytest

import support as S
from ntsc_crt_b200 import layout

pytestmark = pytest.mark.gpu
V = "ntsc_conv"


def trio(outw, outh, fmt=layout.PIX_BGRA):
    gpu = S.ProductEngine(V, outw, outh, fmt)
    ora = S.OracleEngine(V, outw, outh, fmt)
    ref = S.ref_engine(V, outw, outh, fmt, seed=1)
    return gpu, ora, ref


def run_all(engines, fn):
    for e in engines:
        if e is not None:
            fn(e)


def check(gpu, ora, ref, what):
    S.assert_same_state(gpu.state(), ora.state(), what + " [gpu vs oracle]")
    S.assert_same_state(gpu.state(), ref.state(), what + " [gpu vs reference]")


@pytest.mark.parametrize("progressive", [True, False])
@pytest.mark.parametrize("size", [(832, 624), (256, 240)])
def test_conv_cli_sequence(progressive, size):
    img = S.lcg_image(256, 240)
    gpu, ora, ref = trio(*size)
    run_all((gpu, ora, ref), lambda e: S.cli_sequence(e, img, 0, progressive, format=layout.PIX_BGRA))
    check(gpu, ora, ref, "conv cli %r p=%d" % (size, progressive))


def test_conv_config2_every_call():
    img = S.rand_image(832, 624, seed=7)
    gpu, ora, ref = trio(832, 624)
    run_all((gpu, ora, ref), lambda e: e.set(blend=1, scanlines=1))
    for it in range(6):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=it & 1,
                                                      frame=(it >> 1) & 1))
        run_all((gpu, ora, ref), lambda e: e.demodulate(0 if it < 3 else 24))
        check(gpu, ora, ref, "conv cfg2 call %d" % it)


@pytest.mark.parametrize("fmt", range(6))
def test_conv_pixel_formats(fmt):
    rgb = S.rand_image(320, 200, bpp=3, seed=fmt)
    img = S.pack_rgb(rgb, fmt)
    gpu, ora, ref = trio(400, 300, fmt)
    run_all((gpu, ora, ref), lambda e: e.set(blend=1, scanlines=0))
    for it in range(3):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=fmt, as_color=1, field=it & 1, frame=0))
        run_all((gpu, ora, ref), lambda e: e.demodulate(5))
        check(gpu, ora, ref, "conv fmt %d call %d" % (fmt, it))


@pytest.mark.parametrize("outw,outh,fmt,blend,scanlines", [
    (1920, 1080, layout.PIX_BGRA, 1, 1),
    (3200, 300, layout.PIX_RGBA, 0, 0),
    (100, 80, layout.PIX_ARGB, 1, 0),      # fewer rows than lines: ordered passes over shared rows
    (100, 80, layout.PIX_ABGR, 0, 0),
    (333, 250, layout.PIX_BGRA, 1, 1),
    (641, 479, layout.PIX_BGR, 1, 1),
    (640, 480, layout.PIX_RGB, 0, 1),
])
def test_conv_output_geometries(outw, outh, fmt, blend, scanlines):
    img = S.rand_image(400, 300, seed=outw)
    gpu, ora, ref = trio(outw, outh, fmt)
    run_all((gpu, ora, ref), lambda e: e.set(blend=blend, scanlines=scanlines))
    for it in range(3):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=it & 1, frame=0))
        run_all((gpu, ora, ref), lambda e: e.demodulate(2 * it))
        check(gpu, ora, ref, "conv geometry %dx%d fmt %d call %d" % (outw, outh, fmt, it))


def test_conv_knobs_and_generic_path():
    """Monitor knobs, then settings far outside the packed (16-bit chroma) path's exact range, which
    k_sync must route to the generic instantiation."""
    img = S.bars_image(300, 200)
    gpu, ora, ref = trio(512, 448)
    run_all((gpu, ora, ref), lambda e: e.set(hue=37, brightness=9, contrast=200, saturation=14, black_point=3,
                                             white_point=90, blend=0, scanlines=1))
    for it in range(4):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=it & 1, field=it & 1,
                                                      frame=(it >> 1) & 1, hue=20 * it, raw=int(it == 2),  # raw + odd field reads row h (crt_ntsc.c:263)
                                                      xoffset=4 * (it & 1), yoffset=it & 1))
        run_all((gpu, ora, ref), lambda e: e.demodulate(3 * it))
        check(gpu, ora, ref, "conv knobs %d" % it)
    run_all((gpu, ora, ref), lambda e: e.set(saturation=4000, contrast=900, brightness=5000, blend=1))
    for it in range(2):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=it, frame=0))
        run_all((gpu, ora, ref), lambda e: e.demodulate(30))
        check(gpu, ora, ref, "conv extreme %d" % it)


@pytest.mark.parametrize("variant", ["ntsc_conv6", "ntsc_conv5", "ntsc_conv4"])
def test_conv_other_kernels(variant):
    """The 6-, 5- and 4-tap kernels of the same reference build option (crt_core.c:86-88, 136-146)."""
    img = S.rand_image(333, 250, seed=len(variant))
    for outw, outh, fmt, blend, scanlines in ((832, 624, layout.PIX_BGRA, 1, 1), (641, 300, layout.PIX_RGB, 1, 0),
                                               (100, 80, layout.PIX_ARGB, 1, 0)):
        gpu = S.ProductEngine(variant, outw, outh, fmt)
        ora = S.OracleEngine(variant, outw, outh, fmt)
        ref = S.ref_engine(variant, outw, outh, fmt, seed=1)
        run_all((gpu, ora, ref), lambda e: e.set(blend=blend, scanlines=scanlines, hue=-20, brightness=11, saturation=13))
        for it in range(4):
            run_all((gpu, ora, ref), lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=it & 1,
                                                          frame=(it >> 1) & 1))
            run_all((gpu, ora, ref), lambda e: e.demodulate(0 if it < 2 else 21))
            check(gpu, ora, ref, "%s %dx%d call %d" % (variant, outw, outh, it))
        run_all((gpu, ora, ref), lambda e: e.set(saturation=3000, contrast=700, brightness=-4500))
        run_all((gpu, ora, ref), lambda e: e.demodulate(9))
        check(gpu, ora, ref, "%s %dx%d extreme" % (variant, outw, outh))


@pytest.mark.parametrize("tma", [1, 0])
def test_conv_batch_matches_oracle(tma):
    """crtx_* batch interface: independent monitors with different knobs and sources, several fields."""
    import torch
    from ntsc_crt_b200 import capi
    n = 5
    b = capi.Batch(V, n)
    b.set_option("tma", tma)
    outs, oras, imgs = [], [], []
    for i in range(n):
        t = torch.zeros(480, 640, 4, dtype=torch.uint8, device="cuda")
        outs.append(t)
        b.set_monitor(i, t, fmt=layout.PIX_BGRA, noise=3 * i, blend=i & 1, scanlines=(i >> 1) & 1,
                      saturation=8 + i, hue=10 * i)
        o = S.OracleEngine(V, 640, 480)
        o.set(blend=i & 1, scanlines=(i >> 1) & 1, saturation=8 + i, hue=10 * i)
        oras.append(o)
        imgs.append(S.rand_image(320 + 16 * i, 240, seed=100 + i))
    b.commit_monitors()
    dimgs = [torch.from_numpy(im).cuda() for im in imgs]
    for it in range(4):
        for i in range(n):
            b.set_source(i, dimgs[i], format=layout.PIX_BGRA, as_color=1, field=it & 1, frame=(it >> 1) & 1)
            oras[i].modulate(imgs[i], format=layout.PIX_BGRA, as_color=1, field=it & 1, frame=(it >> 1) & 1)
            oras[i].demodulate(3 * i)
        b.modulate()
        b.demodulate()
        torch.cuda.synchronize()
        for i in range(n):
            got = outs[i].cpu().numpy()
            assert np.array_equal(got, oras[i].out), "conv batch monitor %d field %d: %s" % (
                i, it, S.diff_report("out", got, oras[i].out))
    b.close()
