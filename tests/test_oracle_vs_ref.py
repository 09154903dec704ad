"""Pin the oracle (oracle/crt_oracle.c) against the reference itself.

The reference has no tests or golden vectors (SURVEY.md section 4), so the pin is the
UNMODIFIED reference compiled into oracle/_ref/libref_*.so by oracle/Makefile.  Every
case drives both through the same call sequence and compares analog / inp / out / ccf /
hsync / vsync / rn bit for bit after every call.  Where oracle/_ref is not built, the
reference's side is what it produced in the same test, recorded under tests/golden/reference/.
"""
import ctypes as C

import numpy as np
import pytest

import support as S
from ntsc_crt_b200 import layout


def pair(variant, outw, outh, fmt=layout.PIX_BGRA, seed=1):
    ref = S.ref_engine(variant, outw, outh, fmt, seed=seed)
    ora = S.OracleEngine(variant, outw, outh, fmt, seed=seed)
    return ref, ora


def both(ref, ora, fn):
    fn(ref)
    fn(ora)


def check(ref, ora, what):
    S.assert_same_state(ref.state(), ora.state(), what)


def ref_layout(variant):
    """struct sizes, geometry and struct CRT offsets the compiled reference reports"""
    lib = C.CDLL(S.ref_path(variant))
    g = (C.c_int * 20)()
    lib.ref_geometry(g)
    o = (C.c_int * 19)()
    lib.ref_crt_offsets(o)
    return dict(sizeof_crt=lib.ref_sizeof_crt(), sizeof_settings=lib.ref_sizeof_settings(), geometry=list(g)[:12],
                offsets=list(o))


def test_struct_layout_matches_reference():
    for variant in ("ntsc", "ntsc_bloom", "ntsc_conv", "ntsc_conv6", "ntsc_conv5", "ntsc_conv4", "vhs", "nes", "nes_p0", "nes_p1", "snes", "nesrgb", "nesrgb_p0", "nesrgb_p1", "template", "pv1k"):
        spec = layout.system_spec(variant)
        ref = S.ref_result(lambda: ref_layout(variant), S.have_ref(variant))
        assert ref["sizeof_crt"] == C.sizeof(layout.crt_struct(spec)), variant
        assert ref["sizeof_settings"] == C.sizeof(layout.settings_struct(spec)), variant
        assert ref["geometry"] == [spec.hres, spec.vres, spec.input_size, spec.top, spec.bot,
                                   spec.vper, spec.cc_samples, spec.sync_beg, spec.bw_beg, spec.cb_beg,
                                   spec.av_beg, spec.av_len], variant
        CRT = layout.crt_struct(spec)
        names = ["analog", "inp", "outw", "outh", "out_format", "out", "hue", "brightness",
                 "contrast", "saturation", "black_point", "white_point", "scanlines", "blend",
                 "v_fac", "ccf", "hsync", "vsync", "rn"]
        assert ref["offsets"] == [getattr(CRT, n).offset for n in names], variant


SINCOS_ARGS = list(range(-20000, 40000, 7)) + [0, 4095, 4096, 8191, 8192, 12288, 16383, 16384]


def sincos_table(fn):
    s, c = C.c_int(), C.c_int()
    out = np.empty((len(SINCOS_ARGS), 2), dtype=np.int32)
    for i, n in enumerate(SINCOS_ARGS):
        fn(C.byref(s), C.byref(c), n)
        out[i] = s.value, c.value
    return out


def test_sincos_and_bpp():
    live = S.have_ref("ntsc")
    lib = layout.bind_crt_api(C.CDLL(S.ref_path("ntsc")), layout.system_spec("ntsc")) if live else None
    ora = S.oracle_lib()
    ours = sincos_table(ora.ocrt_sincos14)
    want = S.ref_result(lambda: S.digest(sincos_table(lib.crt_sincos14)), live)
    if live:
        theirs = sincos_table(lib.crt_sincos14)
        bad = np.argwhere((theirs != ours).any(axis=1))
        assert not len(bad), SINCOS_ARGS[int(bad[0][0])]
    assert S.digest(ours) == want
    bpp = S.ref_result(lambda: [lib.crt_bpp4fmt(f) for f in range(-2, 9)], live)
    assert bpp == [ora.ocrt_bpp(f) for f in range(-2, 9)] == [layout.bpp4fmt(f) for f in range(-2, 9)]


def test_rand_replica_matches_glibc():
    live = S.have_ref("vhs")
    lib = C.CDLL(S.ref_path("vhs")) if live else None
    ora = S.oracle_lib()
    g = S._ORand()

    def ref_stream(seed):
        lib.ref_srand.argtypes = [C.c_uint]
        lib.ref_srand(seed)
        return np.array([lib.ref_rand() for _ in range(2000)], dtype=np.int64)

    for seed in (1, 0, 42, 2**31 + 5, 0xFFFFFFFF):
        ora.ocrt_rand_seed(C.byref(g), seed)
        ours = np.array([ora.ocrt_rand_next(C.byref(g)) for _ in range(2000)], dtype=np.int64)
        assert S.digest(ours) == S.ref_result(lambda: S.digest(ref_stream(seed)), live), seed


def test_system_coefficients():
    """eq / iir constants quoted in SURVEY.md 8a (probed from the compiled reference)."""
    ora = S.oracle_lib()
    nt = ora.ocrt_system(0, 1).contents
    assert [list(r) for r in nt.eq] == [[42156, 79824, 65536, 8192, 9175],
                                        [2252, 32636, 65536, 65536, 1311],
                                        [2252, 28248, 65536, 65536, 0]]
    assert list(nt.iir_c) == [1233, 574, 232]
    assert list(ora.ocrt_system(5, 1).contents.iir_c) == [987, 262, 262]


@pytest.mark.parametrize("progressive", [True, False])
def test_ntsc_cli_sequence_config1(progressive):
    """config 1: 256x240 in, noise 0 -> 832x624 and 256x240 (crt_main.c:221-255)."""
    img = S.lcg_image(256, 240)
    for outw, outh in ((832, 624), (256, 240)):
        ref, ora = pair("ntsc", outw, outh)
        both(ref, ora, lambda e: S.cli_sequence(e, img, 0, progressive, format=layout.PIX_BGRA))
        check(ref, ora, "cfg1 %dx%d p=%d" % (outw, outh, progressive))


def test_ntsc_every_call_config2():
    """config 2: 832x624 interlaced colour, compare after every single call."""
    img = S.rand_image(832, 624, seed=7)
    ref, ora = pair("ntsc", 832, 624)
    both(ref, ora, lambda e: e.set(blend=1, scanlines=1))
    f, fr = 0, 0
    for it in range(8):
        both(ref, ora, lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=f, frame=fr))
        check(ref, ora, "mod %d" % it)
        both(ref, ora, lambda e: e.demodulate(0))
        check(ref, ora, "demod %d" % it)
        f ^= 1
        if it % 2 == 1:
            fr ^= 1


@pytest.mark.parametrize("noise", [12, 24, 255])
def test_ntsc_noise(noise):
    img = S.bars_image(640, 480)
    ref, ora = pair("ntsc", 640, 480)
    both(ref, ora, lambda e: e.set(blend=0, scanlines=1))
    for it in range(6):
        both(ref, ora, lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=it & 1,
                                            frame=(it >> 1) & 1))
        both(ref, ora, lambda e: e.demodulate(noise))
        check(ref, ora, "noise %d call %d" % (noise, it))


@pytest.mark.parametrize("fmt", range(6))
def test_ntsc_pixel_formats(fmt):
    rgb = S.rand_image(320, 200, bpp=3, seed=fmt)
    img = S.pack_rgb(rgb, fmt)
    ref, ora = pair("ntsc", 400, 300, fmt)
    both(ref, ora, lambda e: e.set(blend=1, scanlines=0))
    for it in range(3):
        both(ref, ora, lambda e: e.modulate(img, format=fmt, as_color=1, field=it & 1, frame=0))
        both(ref, ora, lambda e: e.demodulate(5))
        check(ref, ora, "fmt %d call %d" % (fmt, it))


def test_ntsc_knobs_raw_mono_offsets():
    img = S.bars_image(300, 200)
    ref, ora = pair("ntsc", 512, 448)
    both(ref, ora, lambda e: e.set(hue=37, brightness=9, contrast=200, saturation=14,
                                   black_point=3, white_point=90, blend=0, scanlines=1))
    cases = [dict(raw=1, as_color=1, hue=20, xoffset=8, yoffset=2),
             dict(raw=0, as_color=0, hue=0, xoffset=0, yoffset=0),
             dict(raw=1, as_color=1, hue=350, xoffset=4, yoffset=1),
             dict(raw=0, as_color=1, hue=90, xoffset=0, yoffset=0)]
    for it, kw in enumerate(cases * 2):
        both(ref, ora, lambda e: e.modulate(img, format=layout.PIX_BGRA, field=it & 1,
                                            frame=(it >> 1) & 1, **kw))
        both(ref, ora, lambda e: e.demodulate(3 * it))
        check(ref, ora, "knobs %d" % it)
    both(ref, ora, lambda e: e.set(hue=-45, saturation=31, contrast=255, brightness=-20))
    both(ref, ora, lambda e: e.demodulate(0))
    check(ref, ora, "negative hue")


def test_ntsc_unknown_format_is_silent_noop():
    img = S.rand_image(64, 48)
    ref, ora = pair("ntsc", 128, 96, 9)
    both(ref, ora, lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1))
    both(ref, ora, lambda e: e.demodulate(4))
    check(ref, ora, "bad out format")
    ref, ora = pair("ntsc", 128, 96)
    both(ref, ora, lambda e: e.modulate(img, format=17, as_color=1))
    check(ref, ora, "bad in format")


@pytest.mark.parametrize("outw,outh,blend,scanlines", [(832, 624, 1, 1), (640, 480, 0, 1), (256, 240, 1, 0),
                                                       (300, 100, 1, 0)])
def test_ntsc_conv_variant(outw, outh, blend, scanlines):
    """a11: the USE_CONVOLUTION 1 build (crt_core.c:85-147, 7-tap kernel) against the oracle's FIR eqf."""
    img = S.rand_image(333, 250, seed=outw)
    ref, ora = pair("ntsc_conv", outw, outh)
    both(ref, ora, lambda e: e.set(blend=blend, scanlines=scanlines, hue=15, brightness=-7, contrast=190,
                                   saturation=12))
    for it in range(5):
        both(ref, ora, lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=it & 1,
                                            frame=(it >> 1) & 1))
        both(ref, ora, lambda e: e.demodulate(0 if it < 2 else 17))
        check(ref, ora, "conv %dx%d call %d" % (outw, outh, it))


@pytest.mark.parametrize("variant", ["ntsc_conv6", "ntsc_conv5", "ntsc_conv4"])
def test_ntsc_conv_other_kernels(variant):
    """the 6-, 5- and 4-tap kernels of the same build option (crt_core.c:86-88, 136-146)"""
    img = S.rand_image(333, 250, seed=len(variant))
    ref, ora = pair(variant, 640, 480)
    both(ref, ora, lambda e: e.set(blend=1, scanlines=1, hue=-20, brightness=11, saturation=13))
    for it in range(4):
        both(ref, ora, lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=it & 1,
                                            frame=(it >> 1) & 1))
        both(ref, ora, lambda e: e.demodulate(0 if it < 2 else 21))
        check(ref, ora, "%s call %d" % (variant, it))
    both(ref, ora, lambda e: e.set(saturation=3000, contrast=700, brightness=-4500))
    both(ref, ora, lambda e: e.demodulate(9))
    check(ref, ora, "%s extreme" % variant)


def test_ntsc_conv_extreme_knobs_and_formats():
    for fmt in range(6):
        rgb = S.rand_image(200, 120, bpp=3, seed=40 + fmt)
        img = S.pack_rgb(rgb, fmt)
        ref, ora = pair("ntsc_conv", 400, 300, fmt)
        both(ref, ora, lambda e: e.set(blend=fmt & 1, scanlines=1, saturation=4000, contrast=900, brightness=5000))
        for it in range(2):
            both(ref, ora, lambda e: e.modulate(img, format=fmt, as_color=1, field=it, frame=0))
            both(ref, ora, lambda e: e.demodulate(30))
            check(ref, ora, "conv extreme fmt %d call %d" % (fmt, it))


@pytest.mark.parametrize("fmt,as_color,raw", [(layout.PIX_BGRA, 1, 0), (layout.PIX_RGB, 1, 0), (layout.PIX_ARGB, 0, 0),
                                              (layout.PIX_ABGR, 1, 1)])
def test_snes(fmt, as_color, raw):
    """SURVEY 8f-3: CRT_SYSTEM_SNES (crt_snes.c): RGB source on the NES line layout, 3-line chroma cycle with
    dot crawl, no encoder band-limit."""
    rgb = S.rand_image(300 if not raw else 200, 230 if not raw else 180, bpp=3, seed=fmt)
    img = S.pack_rgb(rgb, fmt)
    ref, ora = pair("snes", 640, 480)
    both(ref, ora, lambda e: e.set(blend=1, scanlines=1, hue=10, saturation=12, black_point=2, white_point=95))
    for it in range(5):
        both(ref, ora, lambda e: e.modulate(img, format=fmt, as_color=as_color, raw=raw, field=it & 1, frame=0,
                                            hue=(it * 50) % 360, dot_crawl_offset=it % 3, xoffset=4 * (it & 1),
                                            yoffset=it % 3))
        check(ref, ora, "snes mod %d" % it)
        both(ref, ora, lambda e: e.demodulate(0 if it < 2 else 9))
        check(ref, ora, "snes demod %d" % it)


@pytest.mark.parametrize("fmt,as_color,raw", [(layout.PIX_BGRA, 1, 0), (layout.PIX_BGR, 1, 0), (layout.PIX_RGBA, 0, 0),
                                              (layout.PIX_ABGR, 1, 1)])
def test_template_system(fmt, as_color, raw):
    """CRT_SYSTEM_TEMP (crt_template.c), the reference's worked example for new systems: NTSC timing, 2-line
    chroma cycle with dot crawl, band-limited, field-dependent sync and source rows.  No product library yet
    (SURVEY 8f-3): this pins the oracle ahead of it."""
    rgb = S.rand_image(300 if not raw else 200, 260 if not raw else 180, bpp=3, seed=fmt)
    img = S.pack_rgb(rgb, fmt)
    ref, ora = pair("template", 640, 480)
    both(ref, ora, lambda e: e.set(blend=1, scanlines=1, hue=-15, saturation=12, black_point=2, white_point=95))
    for it in range(6):
        both(ref, ora, lambda e: e.modulate(img, format=fmt, as_color=as_color, raw=raw, field=it & 1 if not raw else 0,
                                            frame=(it >> 1) & 1, hue=(it * 50) % 360, dot_crawl_offset=it % 4,
                                            xoffset=4 * (it & 1), yoffset=it % 3))
        check(ref, ora, "template mod %d" % it)
        both(ref, ora, lambda e: e.demodulate(0 if it < 2 else 9))
        check(ref, ora, "template demod %d" % it)


@pytest.mark.parametrize("fmt,as_color,raw,conv", [(layout.PIX_BGRA, 1, 0, False), (layout.PIX_RGB, 1, 0, False),
                                                   (layout.PIX_ARGB, 0, 0, False), (layout.PIX_ABGR, 1, 1, False)])
def test_pv1k_system(fmt, as_color, raw, conv):
    """CRT_SYSTEM_PV1K (crt_pv1k.c and the CRT_CC_SAMPLES == 5 branches of crt_core.c:459-467, 480-509, 545-549):
    1920 samples per line, 5 samples per chroma period, separate I / Q carrier tables.  No product library yet
    (SURVEY 8f-3): this pins the oracle ahead of it."""
    rgb = S.rand_image(300 if not raw else 200, 260 if not raw else 180, bpp=3, seed=fmt)
    img = S.pack_rgb(rgb, fmt)
    ref, ora = pair("pv1k", 640, 480)
    both(ref, ora, lambda e: e.set(blend=1, scanlines=1, hue=25, saturation=12, black_point=2, white_point=95))
    for it in range(6):
        both(ref, ora, lambda e: e.modulate(img, format=fmt, as_color=as_color, raw=raw, field=it & 1 if not raw else 0,
                                            frame=(it >> 1) & 1, hue=(it * 50) % 360, dot_crawl_offset=it % 5,
                                            xoffset=5 * (it & 1), yoffset=it % 3))
        check(ref, ora, "pv1k mod %d" % it)
        both(ref, ora, lambda e: e.demodulate(0 if it < 2 else 9))
        check(ref, ora, "pv1k demod %d" % it)


@pytest.mark.parametrize("outw,outh,raw", [(832, 624, 0), (640, 480, 0), (333, 250, 1)])
def test_bloom_option(outw, outh, raw):
    """CRT_DO_BLOOM 1 (crt_core.h:70; crt_core.c:399-402, 512-526; crt_ntsc.c:148-161): a line's width follows the
    filtered beam energy, carried from line to line.  No product library yet (SURVEY 8f-4): this pins the oracle."""
    img = S.bars_image(300, 260) if not raw else S.rand_image(200, 180, seed=5)
    ref, ora = pair("ntsc_bloom", outw, outh)
    both(ref, ora, lambda e: e.set(blend=1, scanlines=1, brightness=4, contrast=190))
    for it in range(5):
        both(ref, ora, lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, raw=raw, field=it & 1 if not raw else 0,
                                            frame=(it >> 1) & 1))
        check(ref, ora, "bloom mod %d" % it)
        both(ref, ora, lambda e: e.demodulate(0 if it < 2 else 20))
        check(ref, ora, "bloom demod %d" % it)


@pytest.mark.parametrize("fmt", [layout.PIX_BGRA, layout.PIX_RGB, layout.PIX_ARGB, 9])
def test_nesrgb(fmt):
    """SURVEY 8f-3: CRT_SYSTEM_NESRGB (crt_nesrgb.c): the NES sync template and burst cycle around an RGB picture.
    Format 9 is unknown: the first call still writes the template, nothing else happens."""
    rgb = S.rand_image(256, 240, bpp=3, seed=3)
    img = S.pack_rgb(rgb, fmt) if fmt != 9 else S.pack_rgb(rgb, layout.PIX_BGRA)
    ref, ora = pair("nesrgb", 640, 480)
    both(ref, ora, lambda e: e.set(blend=0, scanlines=1, saturation=11, black_point=1, white_point=97))
    for it in range(4):
        both(ref, ora, lambda e: e.modulate(img, format=fmt, hue=(it * 70) % 360, dot_crawl_offset=it % 3,
                                            xoffset=4 * (it & 1), yoffset=it % 2))
        check(ref, ora, "nesrgb mod %d" % it)
        both(ref, ora, lambda e: e.demodulate(0 if it < 2 else 7))
        check(ref, ora, "nesrgb demod %d" % it)


@pytest.mark.parametrize("variant", ["nesrgb_p0", "nesrgb_p1"])
def test_nesrgb_chroma_patterns(variant):
    """the NES-RGB system with the other two chroma patterns of crt_nesrgb.h:27-40 (912 / 910 samples per line)"""
    img = S.rand_image(256, 240, seed=8)
    ref, ora = pair(variant, 832, 624)
    both(ref, ora, lambda e: e.set(blend=1, scanlines=1, saturation=12))
    for it in range(4):
        both(ref, ora, lambda e: e.modulate(img, format=layout.PIX_BGRA, hue=(it * 70) % 360, dot_crawl_offset=it % 3,
                                            xoffset=4 * (it & 1), yoffset=it % 2))
        check(ref, ora, "%s mod %d" % (variant, it))
        both(ref, ora, lambda e: e.demodulate(0 if it < 2 else 7))
        check(ref, ora, "%s demod %d" % (variant, it))


@pytest.mark.parametrize("variant", ["nes", "nes_p0", "nes_p1"])
def test_nes(variant):
    """config 3: NES PPU pixels, dot crawl cycling 0,1,2 (crt_main.c:471)."""
    for img in (S.nes_image(seed=5), S.nes_image(rainbow=True)):
        ref, ora = pair(variant, 832, 624)
        both(ref, ora, lambda e: e.set(blend=0, scanlines=1))
        for it in range(5):
            both(ref, ora, lambda e: e.modulate(img, dot_crawl_offset=it % 3, hue=(it * 30) % 360))
            check(ref, ora, "%s mod %d" % (variant, it))
            both(ref, ora, lambda e: e.demodulate(it * 4))
            check(ref, ora, "%s demod %d" % (variant, it))


@pytest.mark.parametrize("color,aberr", [(1, 0), (0, 0), (1, 1)])
def test_vhs(color, aberr):
    """config 5: VHS 832x624 noise 24 (libc rand() stream seeded identically).

    With do_aberration the bottom lines lose their sync pulse, hsync runs away and the
    reference reads its decode window PAST inp[] into the rest of struct CRT (which holds
    an ASLR-dependent pointer): those output rows are outside the parity domain
    (SURVEY.md 7.3-6) and are masked; blend=0 keeps them from leaking into later fields.
    """
    img = S.bars_image(832, 624)
    ref, ora = pair("vhs", 832, 624, seed=1)
    both(ref, ora, lambda e: e.set(blend=0 if aberr else 1, scanlines=1))
    for it in range(4):
        both(ref, ora, lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=color,
                                            field=it & 1, frame=(it >> 1) & 1, do_aberration=aberr))
        check(ref, ora, "vhs mod %d" % it)
        ref.demodulate(24)
        ora.noise_pass(24)
        _, table = ora.sync_pass()
        ora.line_pass(table)
        a, b = ref.state(), ora.state()
        for rec in table:
            if not rec.skip and rec.pos + ora.spec.av_len > ora.spec.input_size:
                assert aberr, "decode window left inp[] without aberration"
                a["out"][rec.beg:rec.end] = 0
                b["out"][rec.beg:rec.end] = 0
                ref.out[rec.beg:rec.end] = 0
                ora.out[rec.beg:rec.end] = 0
        S.assert_same_state(a, b, "vhs demod %d" % it)


def test_staged_decode_equals_whole_decode():
    """The oracle's three-stage split (what the kernels mirror) is the same function."""
    img = S.bars_image(400, 300)
    a = S.OracleEngine("ntsc", 640, 480)
    b = S.OracleEngine("ntsc", 640, 480)
    for e in (a, b):
        e.set(blend=1, scanlines=1)
    for it in range(3):
        for e in (a, b):
            e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=it & 1, frame=0)
        a.demodulate(10)
        b.noise_pass(10)
        _, table = b.sync_pass()
        b.line_pass(table, 0, 100)
        b.line_pass(table, 100, 140)
        S.assert_same_state(a.state(), b.state(), "staged %d" % it)


def test_lcg_jump():
    ora = S.oracle_lib()
    m, a = C.c_uint(), C.c_uint()
    ora.ocrt_lcg_jump(238420, C.byref(m), C.byref(a))
    assert (m.value, a.value) == (0x5535B491, 0xF58BFA78)  # SURVEY.md 7.2 K1 probe
