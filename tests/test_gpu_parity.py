"""GPU parity: the CUDA product library against the oracle and the reference (compiled in oracle/_ref, else its
states recorded under tests/golden/reference/), bit for bit, through the C-ABI.

Two layers:
  * drop-in: the reference's own interface (crt_init / crt_modulate / crt_demodulate on host
    buffers), same call sequences as tests/test_oracle_vs_ref.py;
  * stages: the crtx_* batch interface, checking each kernel's output on its own (analog after
    modulate, inp after the noise pass, the per-line sync table, the decoded image).
"""
import numpy as np
import pytest

import support as S
from ntsc_crt_b200 import layout

pytestmark = pytest.mark.gpu


def trio(variant, outw, outh, fmt=layout.PIX_BGRA):
    gpu = S.ProductEngine(variant, outw, outh, fmt)
    ora = S.OracleEngine(variant, outw, outh, fmt)
    ref = S.ref_engine(variant, outw, outh, fmt, seed=1)
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
def test_dropin_ntsc_config1(progressive, size):
    """config 1: 256x240 in, noise 0, the CLI accumulate loop (crt_main.c:221-255)."""
    img = S.lcg_image(256, 240)
    gpu, ora, ref = trio("ntsc", *size)
    run_all((gpu, ora, ref), lambda e: S.cli_sequence(e, img, 0, progressive, format=layout.PIX_BGRA))
    check(gpu, ora, ref, "cfg1 %r p=%d" % (size, progressive))


def test_dropin_ntsc_config2_every_call():
    """config 2: 832x624 interlaced full colour, compared after every single call."""
    img = S.rand_image(832, 624, seed=7)
    gpu, ora, ref = trio("ntsc", 832, 624)
    run_all((gpu, ora, ref), lambda e: e.set(blend=1, scanlines=1))
    f, fr = 0, 0
    for it in range(8):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=f, frame=fr))
        check(gpu, ora, ref, "mod %d" % it)
        run_all((gpu, ora, ref), lambda e: e.demodulate(0))
        check(gpu, ora, ref, "demod %d" % it)
        f ^= 1
        if it % 2 == 1:
            fr ^= 1


@pytest.mark.parametrize("noise", [12, 24, 255])
def test_dropin_ntsc_noise(noise):
    img = S.bars_image(640, 480)
    gpu, ora, ref = trio("ntsc", 640, 480)
    run_all((gpu, ora, ref), lambda e: e.set(blend=0, scanlines=1))
    for it in range(6):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1,
                                                      field=it & 1, frame=(it >> 1) & 1))
        run_all((gpu, ora, ref), lambda e: e.demodulate(noise))
        check(gpu, ora, ref, "noise %d call %d" % (noise, it))


@pytest.mark.parametrize("fmt", range(6))
def test_dropin_ntsc_pixel_formats(fmt):
    rgb = S.rand_image(320, 200, bpp=3, seed=fmt)
    img = S.pack_rgb(rgb, fmt)
    gpu, ora, ref = trio("ntsc", 400, 300, fmt)
    run_all((gpu, ora, ref), lambda e: e.set(blend=1, scanlines=0))
    for it in range(3):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=fmt, as_color=1, field=it & 1, frame=0))
        run_all((gpu, ora, ref), lambda e: e.demodulate(5))
        check(gpu, ora, ref, "fmt %d call %d" % (fmt, it))


@pytest.mark.parametrize("variant", ["ntsc", "nes", "pv1k"])
def test_burst_lock_from_poked_accumulators(variant):
    """crt->ccf is a public field (crt_core.h:74-92) and only the encoders re-prime it: accumulators far from the lock
    value, of either sign, beyond the range in which the kernel's shortcut for x * 127 / 128 holds (2^23) and changing
    sign on the way down must decay exactly as in the reference (crt_core.c:462-467), call after call"""
    nes = variant == "nes"
    img = S.nes_image(seed=11) if nes else S.rand_image(256, 240, seed=11)
    gpu, ora, ref = trio(variant, 400, 300)
    run_all((gpu, ora, ref), lambda e: e.set(blend=0, scanlines=1))
    kw = dict(dot_crawl_offset=1) if nes else dict(format=layout.PIX_BGRA, as_color=1, field=0, frame=0)
    run_all((gpu, ora, ref), lambda e: e.modulate(img, **kw))
    vals = [9000000, -9000000, 16000000, -1, -16000000]

    def poke(e):
        if isinstance(e, S.ReplayedRefEngine):  # (nothing to poke: its states are recorded)
            return
        tab = e.crt.ccf if hasattr(e, "crt") else e.mon.ccf
        for r in range(e.spec.vper):
            for x in range(e.spec.cc_samples):
                tab[r][x] = vals[(r + x) % len(vals)] - 12345 * r
    run_all((gpu, ora, ref), poke)
    for it in range(3):
        run_all((gpu, ora, ref), lambda e: e.demodulate(0 if it == 0 else 7))
        check(gpu, ora, ref, "%s poked ccf, call %d" % (variant, it))


@pytest.mark.parametrize("fmt", [layout.PIX_BGRA, layout.PIX_RGB, layout.PIX_ARGB])
def test_pv1k_staged_encoder_offsets_and_formats(fmt):
    """the PV-1000 takes the staged encoder since round 2 (five carrier phases from shared-memory tables, crt_pv1k.c:262-318):
    x offsets of either parity (the picture then starts on an odd or an even sample: 2-byte or byte stores), raw and scaled
    pictures, colour and monochrome, walking dot-crawl rows, 3- and 4-byte sources"""
    rgb = S.rand_image(300, 200, bpp=3, seed=21)
    img = S.pack_rgb(rgb, fmt)
    gpu, ora, ref = trio("pv1k", 512, 384)
    run_all((gpu, ora, ref), lambda e: e.set(blend=0, scanlines=0, saturation=12))
    cases = [dict(xoffset=0, raw=0, as_color=1), dict(xoffset=1, raw=0, as_color=1), dict(xoffset=3, raw=1, as_color=1),
             dict(xoffset=5, raw=0, as_color=0), dict(xoffset=7, raw=1, as_color=1), dict(xoffset=2, raw=0, as_color=1)]
    for it, kw in enumerate(cases):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=fmt, field=it & 1, frame=0, dot_crawl_offset=it, **kw))
        run_all((gpu, ora, ref), lambda e: e.demodulate(2 * it))
        check(gpu, ora, ref, "pv1k fmt %d case %d %r" % (fmt, it, kw))


@pytest.mark.parametrize("variant", ["ntsc", "nes"])
def test_poked_signal_extremes(variant):
    """crt->analog is the caller's to poke (crt_main.c:430 clears it): -128 -- which no encoder writes, and which the
    noise pass alone turns into -127 (crt_core.c:363-364) -- and +-127 / +-126, scattered over the picture area of a dozen
    lines and the last bytes of the buffer (the copy's partial 16-byte vector), at noise 0 (the packed-byte clamp of
    crt_sync.cuh) and with noise"""
    nes = variant == "nes"
    img = S.nes_image(seed=3) if nes else S.rand_image(256, 240, seed=3)
    gpu, ora, ref = trio(variant, 400, 300)
    run_all((gpu, ora, ref), lambda e: e.set(blend=0, scanlines=0))
    kw = dict(dot_crawl_offset=2) if nes else dict(format=layout.PIX_BGRA, as_color=1, field=0, frame=0)
    n = gpu.spec.input_size
    h = gpu.spec.hres
    rng = np.random.default_rng(17)
    pos = np.concatenate([line * h + rng.integers(300, 800, size=60) for line in range(40, 220, 15)] + [np.arange(n - 21, n)])
    vals = rng.choice(np.array([-128, -128, -127, 127, 126, -126, 0], dtype=np.int8), size=pos.size)

    def poke(e):
        if isinstance(e, S.ReplayedRefEngine):
            return
        if hasattr(e, "crt"):
            buf = np.frombuffer(e.crt, dtype=np.int8, count=n, offset=0)  # analog[] leads the struct (crt_core.h:74-92)
        else:
            buf = np.ctypeslib.as_array(e.mon.analog, shape=(n,)).view(np.int8)
        buf[pos] = vals
    for it, noise in enumerate((0, 9, 0)):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, **kw))
        run_all((gpu, ora, ref), poke)
        run_all((gpu, ora, ref), lambda e: e.demodulate(noise))
        check(gpu, ora, ref, "%s poked analog, call %d (noise %d)" % (variant, it, noise))
    assert (gpu.inp >= -127).all() and (gpu.inp[pos[vals == -128]] == -127).any()


def test_dropin_ntsc_knobs_raw_mono_offsets():
    img = S.bars_image(300, 200)
    gpu, ora, ref = trio("ntsc", 512, 448)
    run_all((gpu, ora, ref), lambda e: e.set(hue=37, brightness=9, contrast=200, saturation=14,
                                             black_point=3, white_point=90, blend=0, scanlines=1))
    cases = [dict(raw=1, as_color=1, hue=20, xoffset=8, yoffset=2),
             dict(raw=0, as_color=0, hue=0, xoffset=0, yoffset=0),
             dict(raw=1, as_color=1, hue=350, xoffset=4, yoffset=1),
             dict(raw=0, as_color=1, hue=90, xoffset=0, yoffset=0)]
    for it, kw in enumerate(cases * 2):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=layout.PIX_BGRA, field=it & 1,
                                                      frame=(it >> 1) & 1, **kw))
        run_all((gpu, ora, ref), lambda e: e.demodulate(3 * it))
        check(gpu, ora, ref, "knobs %d" % it)
    # saturation 31 leaves the fast equaliser path's guaranteed range on some lines
    run_all((gpu, ora, ref), lambda e: e.set(hue=-45, saturation=31, contrast=255, brightness=-20))
    run_all((gpu, ora, ref), lambda e: e.demodulate(0))
    check(gpu, ora, ref, "negative hue, high saturation")
    run_all((gpu, ora, ref), lambda e: e.set(saturation=400, brightness=5000))
    run_all((gpu, ora, ref), lambda e: e.demodulate(2))
    check(gpu, ora, ref, "wrapping saturation / brightness (generic equaliser path)")


def test_dropin_unknown_format_is_silent_noop():
    img = S.rand_image(64, 48)
    gpu, ora, ref = trio("ntsc", 128, 96, 9)
    run_all((gpu, ora, ref), lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1))
    run_all((gpu, ora, ref), lambda e: e.demodulate(4))
    check(gpu, ora, ref, "bad out format")
    gpu, ora, ref = trio("ntsc", 128, 96)
    run_all((gpu, ora, ref), lambda e: e.modulate(img, format=17, as_color=1))
    check(gpu, ora, ref, "bad in format")


@pytest.mark.parametrize("fmt,as_color,raw,outw,outh", [(layout.PIX_BGRA, 1, 0, 832, 624), (layout.PIX_RGB, 1, 0, 640, 480),
                                                        (layout.PIX_ARGB, 0, 0, 333, 250), (layout.PIX_ABGR, 1, 1, 100, 80)])
def test_dropin_snes(fmt, as_color, raw, outw, outh):
    """SURVEY 8f-3: CRT_SYSTEM_SNES (crt_snes.c:125-327) through the drop-in interface."""
    rgb = S.rand_image(300 if not raw else 200, 230 if not raw else 180, bpp=3, seed=fmt)
    img = S.pack_rgb(rgb, fmt)
    gpu, ora, ref = trio("snes", outw, outh, fmt)
    run_all((gpu, ora, ref), lambda e: e.set(blend=1, scanlines=1, hue=10, saturation=12, black_point=2, white_point=95))
    for it in range(5):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=fmt, as_color=as_color, raw=raw, field=it & 1, frame=0,
                                                      hue=(it * 50) % 360, dot_crawl_offset=it % 3, xoffset=4 * (it & 1),
                                                      yoffset=it % 3))
        check(gpu, ora, ref, "snes mod %d" % it)
        run_all((gpu, ora, ref), lambda e: e.demodulate(0 if it < 2 else 9))
        check(gpu, ora, ref, "snes demod %d" % it)


@pytest.mark.parametrize("fmt,outw,outh", [(layout.PIX_BGRA, 832, 624), (layout.PIX_RGB, 640, 480), (layout.PIX_ARGB, 333, 250),
                                           (9, 320, 240)])
def test_dropin_nesrgb(fmt, outw, outh):
    """SURVEY 8f-3: CRT_SYSTEM_NESRGB (crt_nesrgb.c:19-172) through the drop-in interface (format 9: unknown)."""
    rgb = S.rand_image(256, 240, bpp=3, seed=3)
    img = S.pack_rgb(rgb, fmt) if fmt != 9 else S.pack_rgb(rgb, layout.PIX_BGRA)
    gpu, ora, ref = trio("nesrgb", outw, outh)
    run_all((gpu, ora, ref), lambda e: e.set(blend=1, scanlines=1, saturation=11, black_point=1, white_point=97))
    for it in range(4):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=fmt, hue=(it * 70) % 360, dot_crawl_offset=it % 3,
                                                      xoffset=4 * (it & 1), yoffset=it % 2))
        check(gpu, ora, ref, "nesrgb mod %d" % it)
        run_all((gpu, ora, ref), lambda e: e.demodulate(0 if it < 2 else 7))
        check(gpu, ora, ref, "nesrgb demod %d" % it)


def test_batch_snes_matches_oracle():
    import torch
    from ntsc_crt_b200 import capi
    n = 3
    b = capi.Batch("snes", n)
    outs, oras, imgs = [], [], []
    for i in range(n):
        t = torch.zeros(480, 640, 4, dtype=torch.uint8, device="cuda")
        outs.append(t)
        b.set_monitor(i, t, fmt=layout.PIX_BGRA, noise=4 * i, blend=i & 1, scanlines=1, saturation=9 + i)
        o = S.OracleEngine("snes", 640, 480)
        o.set(blend=i & 1, scanlines=1, saturation=9 + i)
        oras.append(o)
        imgs.append(S.rand_image(256 + 32 * i, 224, seed=200 + i))
    b.commit_monitors()
    dimgs = [torch.from_numpy(im).cuda() for im in imgs]
    for it in range(4):
        for i in range(n):
            kw = dict(format=layout.PIX_BGRA, as_color=1, hue=15 * i, dot_crawl_offset=(it + i) % 3)
            b.set_source(i, dimgs[i], **kw)
            oras[i].modulate(imgs[i], **kw)
            oras[i].demodulate(4 * i)
        b.modulate()
        b.demodulate()
        torch.cuda.synchronize()
        for i in range(n):
            got = outs[i].cpu().numpy()
            assert np.array_equal(got, oras[i].out), "snes batch monitor %d field %d: %s" % (
                i, it, S.diff_report("out", got, oras[i].out))
    b.close()


@pytest.mark.parametrize("variant", ["nes", "nes_p0"])
def test_dropin_nes(variant):
    """config 3: NES PPU pixels incl. CRT_CHROMA_PATTERN 0, dot crawl cycling 0,1,2."""
    for img in (S.nes_image(seed=5), S.nes_image(rainbow=True)):
        gpu, ora, ref = trio(variant, 832, 624)
        run_all((gpu, ora, ref), lambda e: e.set(blend=0, scanlines=1))
        for it in range(5):
            run_all((gpu, ora, ref), lambda e: e.modulate(img, dot_crawl_offset=it % 3, hue=(it * 30) % 360))
            check(gpu, ora, ref, "%s mod %d" % (variant, it))
            run_all((gpu, ora, ref), lambda e: e.demodulate(it * 4))
            check(gpu, ora, ref, "%s demod %d" % (variant, it))


@pytest.mark.parametrize("color", [1, 0])
def test_dropin_vhs(color):
    """config 5: VHS 832x624 noise 24; the drop-in draws from libc rand() like the reference, so the
    comparison is against the oracle's replica of glibc's rand() with the same seed (pinned to the reference by
    tests/test_oracle_vs_ref.py::test_rand_replica_matches_glibc)."""
    import ctypes as C
    img = S.bars_image(832, 624)
    libc = C.CDLL(None)
    gpu = S.ProductEngine("vhs", 832, 624)
    ora = S.OracleEngine("vhs", 832, 624, seed=1)
    gpu.set(blend=1, scanlines=1)
    ora.set(blend=1, scanlines=1)
    libc.srand(1)
    for it in range(4):
        for e in (gpu, ora):
            e.modulate(img, format=layout.PIX_BGRA, as_color=color, field=it & 1, frame=(it >> 1) & 1)
        S.assert_same_state(gpu.state(), ora.state(), "vhs mod %d" % it)
        for e in (gpu, ora):
            e.demodulate(24)
        S.assert_same_state(gpu.state(), ora.state(), "vhs demod %d" % it)


def test_tma_and_plain_staging_agree():
    """The TMA (cp.async.bulk) staging of the line kernel against plain loads, same kernel."""
    import torch
    from ntsc_crt_b200 import capi
    img = torch.from_numpy(S.rand_image(832, 624, seed=11)).cuda()
    outs = []
    for tma in (1, 0):
        b = capi.Batch("ntsc", 2)
        b.set_option("tma", tma)
        o = [torch.zeros(624, 832, 4, dtype=torch.uint8, device="cuda") for _ in range(2)]
        for i in range(2):
            b.set_monitor(i, o[i], noise=7 * i, blend=1, scanlines=1)
            b.set_source(i, img, format=layout.PIX_BGRA, as_color=1, field=i, frame=0)
        b.commit_monitors()
        for _ in range(2):
            b.modulate()
            b.demodulate()
        torch.cuda.synchronize()
        outs.append([x.cpu().numpy() for x in o])
        b.close()
    for i in range(2):
        assert np.array_equal(outs[0][i], outs[1][i])
    assert outs[0][0].any()


def test_batch_matches_independent_oracles():
    """crtx batch of 5 monitors with different knobs / noise = 5 independent reference instances."""
    import torch
    from ntsc_crt_b200 import capi
    n = 5
    imgs = [S.rand_image(200 + 40 * i, 150 + 30 * i, seed=i) for i in range(n)]
    b = capi.Batch("ntsc", n)
    outs = [torch.zeros(480, 640, 4, dtype=torch.uint8, device="cuda") for _ in range(n)]
    dimg = [torch.from_numpy(x).cuda() for x in imgs]
    oras = []
    for i in range(n):
        knobs = dict(hue=10 * i, saturation=8 + i, contrast=170 + 5 * i, blend=i & 1, scanlines=1)
        b.set_monitor(i, outs[i], noise=6 * i, **knobs)
        o = S.OracleEngine("ntsc", 640, 480)
        o.set(**knobs)
        oras.append(o)
    b.commit_monitors()
    for step in range(3):
        for i in range(n):
            b.set_source(i, dimg[i], format=layout.PIX_BGRA, as_color=1, field=step & 1, frame=0)
        b.modulate()
        b.demodulate()
        for i in range(n):
            oras[i].modulate(imgs[i], format=layout.PIX_BGRA, as_color=1, field=step & 1, frame=0)
            oras[i].demodulate(6 * i)
        torch.cuda.synchronize()
        st = b.get_state()
        for i in range(n):
            got = dict(analog=b.signal(i, "analog"), inp=b.signal(i, "inp"), out=outs[i].cpu().numpy(),
                       ccf=np.array([[st[i].ccf[r][x] for x in range(4)] for r in range(1)]),
                       hsync=st[i].hsync, vsync=st[i].vsync, rn=st[i].rn)
            S.assert_same_state(got, oras[i].state(), "batch monitor %d step %d" % (i, step))
    assert b.launches >= 3 * 5  # modulate 2-3, noise, sync, line kernel per geometry group
    b.close()


@pytest.mark.parametrize("outw,outh,fmt,blend,scanlines", [
    (1920, 1080, layout.PIX_BGRA, 1, 1),   # > 2 pixels per sample
    (3200, 300, layout.PIX_RGBA, 0, 0),    # > 4 pixels per sample (dx < 1024)
    (100, 80, layout.PIX_ARGB, 1, 0),      # heavy decimation, fewer rows than lines (lines skipped / shared)
    (333, 250, layout.PIX_BGRA, 1, 1),     # width not a multiple of 4: scalar flush path
    (641, 479, layout.PIX_BGR, 1, 1),      # 3-byte pixels, odd geometry, blend
    (832, 624, layout.PIX_ABGR, 0, 1),
])
def test_dropin_ntsc_output_geometries(outw, outh, fmt, blend, scanlines):
    """Output sizes / formats that take the other flush paths and many-pixels-per-sample resampling."""
    img = S.rand_image(400, 300, seed=outw)
    gpu, ora, ref = trio("ntsc", outw, outh, fmt)
    run_all((gpu, ora, ref), lambda e: e.set(blend=blend, scanlines=scanlines))
    for it in range(3):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=layout.PIX_BGRA, as_color=1, field=it & 1, frame=0))
        run_all((gpu, ora, ref), lambda e: e.demodulate(2 * it))
        check(gpu, ora, ref, "geometry %dx%d fmt %d call %d" % (outw, outh, fmt, it))


@pytest.mark.parametrize("w,h,fmt", [(1920, 1080, layout.PIX_BGRA), (3000, 200, layout.PIX_RGB), (97, 61, layout.PIX_RGBA),
                                     (753, 240, layout.PIX_ARGB)])  # h = 236 would read row h in the reference (crt_ntsc.c:263)
def test_dropin_ntsc_source_geometries(w, h, fmt):
    """Source sizes on both sides of the staged encoder's span limit (wide sources take the gather kernel)."""
    img = S.pack_rgb(S.rand_image(w, h, bpp=3, seed=w), fmt)
    gpu, ora, ref = trio("ntsc", 640, 480)
    run_all((gpu, ora, ref), lambda e: e.set(blend=0, scanlines=1))
    for it in range(2):
        run_all((gpu, ora, ref), lambda e: e.modulate(img, format=fmt, as_color=1, field=it & 1, frame=it))
        check(gpu, ora, ref, "source %dx%d mod %d" % (w, h, it))
        run_all((gpu, ora, ref), lambda e: e.demodulate(0))
        check(gpu, ora, ref, "source %dx%d demod %d" % (w, h, it))


def test_batch_vhs_device_rand_replica_matches_glibc_stream():
    """config 5 in the batch interface: noise and aberration draws come from the per-monitor replica of
    glibc's rand() (crtx_seed), in the reference's draw order -- compared with the oracle driven by the
    same seeds (which tests/test_oracle_vs_ref.py pins against the real libc stream)."""
    import torch
    from ntsc_crt_b200 import capi
    n = 3
    seeds = [1, 42, 2024]
    img = S.bars_image(832, 624)
    dimg = torch.from_numpy(img).cuda()
    b = capi.Batch("vhs", n)
    outs = [torch.zeros(624, 832, 4, dtype=torch.uint8, device="cuda") for _ in range(n)]
    oras = []
    for i in range(n):
        b.set_monitor(i, outs[i], noise=24, blend=1, scanlines=1)
        b.seed(seeds[i], first=i, count=1)
        o = S.OracleEngine("vhs", 832, 624, seed=seeds[i])
        o.set(blend=1, scanlines=1)
        oras.append(o)
    b.commit_monitors()
    for step in range(4):
        aberr = 1 if step == 2 else 0
        for i in range(n):
            b.set_source(i, dimg, format=layout.PIX_BGRA, as_color=1 - (i & 1), field=step & 1, frame=(step >> 1) & 1,
                         do_aberration=aberr)
            oras[i].modulate(img, format=layout.PIX_BGRA, as_color=1 - (i & 1), field=step & 1, frame=(step >> 1) & 1,
                             do_aberration=aberr)
        b.modulate()
        b.demodulate()
        for i in range(n):
            oras[i].demodulate(24)
        torch.cuda.synchronize()
        st = b.get_state()
        for i in range(n):
            got = dict(analog=b.signal(i, "analog"), inp=b.signal(i, "inp"), out=outs[i].cpu().numpy(),
                       ccf=np.array([[st[i].ccf[0][x] for x in range(4)]]),
                       hsync=st[i].hsync, vsync=st[i].vsync, rn=st[i].rn)
            S.assert_same_state(got, oras[i].state(), "vhs batch monitor %d step %d" % (i, step))
    b.close()
