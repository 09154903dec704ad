"""Test support: three interchangeable engines over the same call sequence.

  RefEngine      the UNMODIFIED reference compiled into oracle/_ref/libref_<variant>.so
  OracleEngine   our CPU restatement, oracle/libcrt_oracle.so
  ProductEngine  the CUDA product library, ntsc-crt_b200/lib/libcrt_b200_<variant>.so,
                 through the same C-ABI as the reference (defined in test files that
                 need it; shares CEngine below)

All of them expose: set(**knobs), modulate(img, **settings), demodulate(noise) and the
state arrays analog / inp / out / ccf / hsync / vsync / rn.

Where the compiled reference is absent (it can only be built next to the reference's
sources), RefEngine and ref_result() replay what the reference produced in the same test,
recorded under tests/golden/reference/ (see ref_result).
"""
import atexit
import ctypes as C
import hashlib
import json
import os

import numpy as np

import pkgload

pkg = pkgload.load()
from ntsc_crt_b200 import layout  # noqa: E402

ROOT = pkg.REPO_ROOT
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")

KNOBS = ("hue", "brightness", "contrast", "saturation", "black_point", "white_point",
         "scanlines", "blend", "v_fac")


def ref_path(variant):
    return os.path.join(REF_DIR, "libref_%s.so" % variant)


def have_ref(variant="ntsc"):
    return os.path.exists(ref_path(variant))


# ----------------------------------------------------------------------------------
# recorded reference results
# ----------------------------------------------------------------------------------

REF_GOLDEN_DIR = os.path.join(ROOT, "tests", "golden", "reference")
# a directory to write the reference results of this run into (tests/golden/reference/ to refresh the goldens)
REF_RECORD_DIR = os.environ.get("CRT_REF_RECORD")

_recorded = {}   # module -> {test: [result, ...]} written at exit when REF_RECORD_DIR is set
_golden = {}     # module -> {test: [result, ...]} loaded from REF_GOLDEN_DIR
_run = None      # the running test: [module, test, position of its next result, results so far]


def begin_test(item):
    """Start the reference results of one run of a pytest item (tests/conftest.py calls it before every test).  They
    are keyed by the file and function that define the test, plus its parameters: tests/test_simt_kernels.py runs the
    GPU tests again under other names and replays the same recordings."""
    global _run
    fn = getattr(item, "function", None)
    if fn is None:
        _run = None
        return
    callspec = getattr(item, "callspec", None)
    test = fn.__name__ + ("[%s]" % callspec.id if callspec is not None else "")
    _run = [os.path.basename(fn.__code__.co_filename), test, 0, []]


def end_test():
    """Close the running test's results; a recording run keeps the first run of every key."""
    global _run
    if _run is not None and REF_RECORD_DIR and _run[3]:
        _recorded.setdefault(_run[0], {}).setdefault(_run[1], _run[3])
    _run = None


def digest(a):
    """short content digest of an array (bytes and shape)"""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()[:16]


def ref_result(compute, live):
    """One result of the compiled reference in the running test, in call order.

    live: the compiled reference this result comes from exists -- compute() is called and its value (anything JSON
    can hold; digest() for arrays) returned, and recorded when CRT_REF_RECORD names a directory.  Otherwise the value
    recorded at the same position of the same test under tests/golden/reference/<test module>.json is returned."""
    assert _run is not None, "ref_result() is called from inside a test function (begin_test() starts its results)"
    module, test, pos, results = _run
    _run[2] = pos + 1
    if live:
        value = json.loads(json.dumps(compute()))
        results.append(value)
        return value
    if module not in _golden:
        path = os.path.join(REF_GOLDEN_DIR, module[:-3] + ".json")
        _golden[module] = json.load(open(path)) if os.path.exists(path) else {}
    seq = _golden[module].get(test)
    assert seq is not None and pos < len(seq), (
        "no recorded reference result %d for %s::%s in tests/golden/reference/ (record it where oracle/_ref is built: "
        "CRT_REF_RECORD=tests/golden/reference pytest ...)" % (pos, module, test))
    return seq[pos]


@atexit.register
def _write_recorded():
    if not (REF_RECORD_DIR and _recorded):
        return
    os.makedirs(REF_RECORD_DIR, exist_ok=True)
    for module, tests in _recorded.items():
        path = os.path.join(REF_RECORD_DIR, module[:-3] + ".json")
        old = json.load(open(path)) if os.path.exists(path) else {}
        old.update(tests)
        with open(path, "w") as f:  # one test per line
            f.write("{\n%s\n}\n" % ",\n".join("%s:%s" % (json.dumps(t), json.dumps(old[t], separators=(",", ":")))
                                               for t in sorted(old)))


# ----------------------------------------------------------------------------------
# synthetic inputs (SURVEY.md 8d): seeded LCG noise, colour bars, 1-px checker, flats
# ----------------------------------------------------------------------------------

def lcg_image(w, h, bpp=4, seed=12345):
    """x = x*1664525 + 1013904223; px = (x >> 8) & 0xffffff (SURVEY.md 8d config 1)."""
    n = w * h
    a, c, m = 1664525, 1013904223, 0xFFFFFFFF
    v = seed & m
    out = np.empty(n, dtype=np.uint32)
    for i in range(n):
        v = (v * a + c) & m
        out[i] = (v >> 8) & 0xFFFFFF
    img = np.zeros((h, w, bpp), dtype=np.uint8)
    img[..., 0] = (out & 0xFF).reshape(h, w)
    img[..., 1] = ((out >> 8) & 0xFF).reshape(h, w)
    img[..., 2] = ((out >> 16) & 0xFF).reshape(h, w)
    if bpp == 4:
        img[..., 3] = 0xFF
    return img


def rand_image(w, h, bpp=4, seed=1):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 256, size=(h, w, bpp), dtype=np.uint8)


def bars_image(w, h, bpp=4, fmt=layout.PIX_BGRA):
    """75% colour bars over a luma ramp and a 1-px checker (artifact colours)."""
    cols = [(191, 191, 191), (191, 191, 0), (0, 191, 191), (0, 191, 0),
            (191, 0, 191), (191, 0, 0), (0, 0, 191), (0, 0, 0)]
    rgb = np.zeros((h, w, 3), dtype=np.uint8)
    for x in range(w):
        rgb[: (2 * h) // 3, x] = cols[min(7, x * 8 // w)]
    ramp = (np.arange(w) * 255 // max(1, w - 1)).astype(np.uint8)
    rgb[(2 * h) // 3: (5 * h) // 6] = ramp[None, :, None]
    yy, xx = np.mgrid[(5 * h) // 6: h, 0:w]
    rgb[(5 * h) // 6:] = (((xx + yy) & 1) * 255).astype(np.uint8)[..., None]
    return pack_rgb(rgb, fmt)


def pack_rgb(rgb, fmt):
    """(h, w, 3) RGB -> (h, w, bpp) in one of the CRT_PIX_FORMATs."""
    h, w, _ = rgb.shape
    bpp = layout.bpp4fmt(fmt)
    out = np.full((h, w, bpp), 0xFF, dtype=np.uint8)
    order = {layout.PIX_RGB: (0, 1, 2), layout.PIX_BGR: (2, 1, 0),
             layout.PIX_ARGB: (1, 2, 3), layout.PIX_RGBA: (0, 1, 2),
             layout.PIX_ABGR: (3, 2, 1), layout.PIX_BGRA: (2, 1, 0)}[fmt]
    for ch, pos in enumerate(order):
        out[..., pos] = rgb[..., ch]
    return out


def nes_image(w=256, h=240, seed=3, rainbow=False):
    """9-bit PPU pixels (crt_nes.c:44-60): hue[3:0] level[5:4] emphasis[8:6]."""
    if rainbow:
        xx = np.arange(w)[None, :] + np.zeros((h, 1), dtype=np.int64)
        yy = np.arange(h)[:, None] + np.zeros((1, w), dtype=np.int64)
        hue = 1 + ((xx + yy // 8) % 12)
        lvl = 1 + ((xx // 16) % 3)
        return (hue | (lvl << 4) | (((yy // 60) % 8) << 6)).astype(np.uint16)
    rng = np.random.default_rng(seed)
    return rng.integers(0, 512, size=(h, w), dtype=np.uint16)


# ----------------------------------------------------------------------------------
# engines
# ----------------------------------------------------------------------------------

class CEngine:
    """Drives any library exporting the reference's C interface (crt_core.h:100-139)."""

    def __init__(self, lib_path, variant, outw, outh, fmt=layout.PIX_BGRA, out=None):
        self.spec = layout.system_spec(variant)
        self.lib = layout.bind_crt_api(C.CDLL(lib_path), self.spec)
        self.CRT = layout.crt_struct(self.spec)
        self.Settings = layout.settings_struct(self.spec)
        self.crt = self.CRT()
        bpp = max(1, layout.bpp4fmt(fmt))
        self.out = out if out is not None else np.zeros((outh, outw, bpp), dtype=np.uint8)
        self.lib.crt_init(C.byref(self.crt), outw, outh, fmt, self.out.ctypes.data)
        self.settings = self.Settings()  # zeroed, as crt_ntsc.h:122 demands
        self._img = None

    def set(self, **kw):
        for k, v in kw.items():
            assert k in KNOBS or k in ("hsync", "vsync", "rn"), k
            setattr(self.crt, k, v)
        return self

    def resize(self, outw, outh, fmt, out):
        self.out = out
        self.lib.crt_resize(C.byref(self.crt), outw, outh, fmt, out.ctypes.data)

    def reset(self):
        self.lib.crt_reset(C.byref(self.crt))

    def modulate(self, img, **kw):
        self._img = np.ascontiguousarray(img)
        s = self.settings
        s.data = self._img.ctypes.data
        s.h, s.w = self._img.shape[0], self._img.shape[1]
        for k, v in kw.items():
            setattr(s, k, v)
        self.lib.crt_modulate(C.byref(self.crt), C.byref(s))

    def demodulate(self, noise=0):
        self.lib.crt_demodulate(C.byref(self.crt), noise)

    @property
    def analog(self):
        return np.frombuffer(self.crt, dtype=np.int8, count=self.spec.input_size, offset=0).copy()

    @property
    def inp(self):
        return np.frombuffer(self.crt, dtype=np.int8, count=self.spec.input_size,
                             offset=self.spec.input_size).copy()

    @property
    def ccf(self):
        return np.array([[self.crt.ccf[n][x] for x in range(self.spec.cc_samples)] for n in range(self.spec.vper)])

    @property
    def hsync(self):
        return self.crt.hsync

    @property
    def vsync(self):
        return self.crt.vsync

    @property
    def rn(self):
        return self.crt.rn

    def state(self):
        return dict(analog=self.analog, inp=self.inp, out=self.out.copy(), ccf=self.ccf,
                    hsync=self.hsync, vsync=self.vsync, rn=self.rn)


class RefState(dict):
    """A state of the reference; `replayed`: it holds no arrays, assert_same_state compares with the recorded digest."""
    replayed = False


STATE_KEYS = ("hsync", "vsync", "rn", "ccf", "analog", "inp", "out")


def state_digest(st):
    return [int(st["hsync"]), int(st["vsync"]), int(st["rn"]), digest(np.asarray(st["ccf"], dtype=np.int64)),
            digest(st["analog"]), digest(st["inp"]), digest(st["out"])]


class RefEngine(CEngine):
    def __init__(self, variant, outw, outh, fmt=layout.PIX_BGRA, out=None, seed=None):
        super().__init__(ref_path(variant), variant, outw, outh, fmt, out)
        self.lib.ref_srand.argtypes = [C.c_uint]
        if seed is not None:
            self.lib.ref_srand(seed)

    def state(self):
        return RefState(super().state())


class ReplayedRefEngine:
    """Stands in for RefEngine where oracle/_ref is not built: takes the same calls and does nothing; its states are
    the ones RefEngine recorded at the same point of the same test (see ref_result)."""

    def __init__(self, variant, outw, outh, fmt=layout.PIX_BGRA, out=None, seed=None):
        self.out = out if out is not None else np.zeros((outh, outw, max(1, layout.bpp4fmt(fmt))), dtype=np.uint8)

    def set(self, **kw):
        return self

    def resize(self, outw, outh, fmt, out):
        self.out = out

    def reset(self):
        pass

    def modulate(self, img, **kw):
        pass

    def demodulate(self, noise=0):
        pass

    def state(self):
        st = RefState(out=self.out.copy())  # (tests may mask rows of it before comparing)
        st.replayed = True
        return st


def ref_engine(variant, outw, outh, fmt=layout.PIX_BGRA, out=None, seed=None):
    """The compiled reference where oracle/_ref has it, else its recorded states."""
    cls = RefEngine if have_ref(variant) else ReplayedRefEngine
    return cls(variant, outw, outh, fmt, out, seed)


class _OSys(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "system", "chroma_pattern", "hres", "vres", "input_size", "top", "bot", "lines",
        "cc_vper", "hsync_window", "vsync_window", "hsync_thresh", "vsync_thresh",
        "sync_beg", "bw_beg", "cb_beg", "av_beg", "av_len", "burst_len",
        "white_level", "burst_level", "black_level", "blank_level", "sync_level",
        "vhs_noise", "nes_vsync_end")] + [("eq", (C.c_int * 5) * 3), ("iir_c", C.c_int * 3), ("conv", C.c_int), ("cc_samples", C.c_int), ("bloom", C.c_int)]


class _OMonitor(C.Structure):
    _fields_ = [
        ("analog", C.POINTER(C.c_byte)), ("inp", C.POINTER(C.c_byte)),
        ("outw", C.c_int), ("outh", C.c_int), ("out_format", C.c_int),
        ("out", C.c_void_p),
        ("hue", C.c_int), ("brightness", C.c_int), ("contrast", C.c_int),
        ("saturation", C.c_int), ("black_point", C.c_int), ("white_point", C.c_int),
        ("scanlines", C.c_int), ("blend", C.c_int), ("v_fac", C.c_uint),
        ("ccf", (C.c_int * 5) * 5), ("hsync", C.c_int), ("vsync", C.c_int), ("rn", C.c_int),
        ("last_noise", C.c_int),
    ]


class _ORgb(C.Structure):
    _fields_ = [("data", C.c_void_p)] + [(n, C.c_int) for n in (
        "format", "w", "h", "raw", "as_color", "field", "frame", "hue", "xoffset",
        "yoffset", "do_aberration", "dot_crawl_offset")]


class _ONes(C.Structure):
    _fields_ = [("data", C.c_void_p)] + [(n, C.c_int) for n in (
        "w", "h", "dot_crawl_offset", "hue", "xoffset", "yoffset", "field_initialized")]


class _ONesRgb(C.Structure):
    _fields_ = [("data", C.c_void_p)] + [(n, C.c_int) for n in (
        "format", "w", "h", "dot_crawl_offset", "hue", "xoffset", "yoffset", "field_initialized")]


class _ORand(C.Structure):
    _fields_ = [("r", C.c_uint * 31), ("f", C.c_int), ("b", C.c_int)]


class OLine(C.Structure):
    _fields_ = [("skip", C.c_int), ("beg", C.c_int), ("end", C.c_int), ("hsync", C.c_int),
                ("pos", C.c_int), ("wave", C.c_int * 4), ("wave_i", C.c_int * 5), ("wave_q", C.c_int * 5)]


_oracle = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        lib = C.CDLL(os.path.join(ORACLE_DIR, "libcrt_oracle.so"))
        lib.ocrt_system.restype = C.POINTER(_OSys)
        lib.ocrt_system.argtypes = [C.c_int, C.c_int]
        lib.ocrt_system_conv.restype = C.POINTER(_OSys)
        lib.ocrt_system_conv.argtypes = [C.c_int, C.c_int]
        lib.ocrt_system_conv_taps.restype = C.POINTER(_OSys)
        lib.ocrt_system_conv_taps.argtypes = [C.c_int, C.c_int, C.c_int]
        lib.ocrt_system_bloom.restype = C.POINTER(_OSys)
        lib.ocrt_system_bloom.argtypes = [C.c_int, C.c_int]
        lib.ocrt_monitor_create.argtypes = [C.POINTER(_OSys), C.POINTER(_OMonitor), C.c_int,
                                            C.c_int, C.c_int, C.c_void_p]
        lib.ocrt_monitor_create.restype = C.c_int
        lib.ocrt_monitor_destroy.argtypes = [C.POINTER(_OMonitor)]
        lib.ocrt_monitor_reset.argtypes = [C.POINTER(_OMonitor)]
        lib.ocrt_encode_rgb.argtypes = [C.POINTER(_OSys), C.POINTER(_OMonitor),
                                        C.POINTER(_ORgb), C.POINTER(_ORand)]
        lib.ocrt_encode_nes.argtypes = [C.POINTER(_OSys), C.POINTER(_OMonitor), C.POINTER(_ONes)]
        lib.ocrt_encode_snes.argtypes = [C.POINTER(_OSys), C.POINTER(_OMonitor), C.POINTER(_ORgb)]
        lib.ocrt_encode_nesrgb.argtypes = [C.POINTER(_OSys), C.POINTER(_OMonitor), C.POINTER(_ONesRgb)]
        lib.ocrt_encode_template.argtypes = [C.POINTER(_OSys), C.POINTER(_OMonitor), C.POINTER(_ORgb)]
        lib.ocrt_encode_pv1k.argtypes = [C.POINTER(_OSys), C.POINTER(_OMonitor), C.POINTER(_ORgb)]
        lib.ocrt_decode.argtypes = [C.POINTER(_OSys), C.POINTER(_OMonitor), C.c_int,
                                    C.POINTER(_ORand)]
        lib.ocrt_noise_pass.argtypes = lib.ocrt_decode.argtypes
        lib.ocrt_sync_pass.argtypes = [C.POINTER(_OSys), C.POINTER(_OMonitor), C.POINTER(OLine)]
        lib.ocrt_sync_pass.restype = C.c_int
        lib.ocrt_line_pass.argtypes = [C.POINTER(_OSys), C.POINTER(_OMonitor), C.POINTER(OLine),
                                       C.c_int, C.c_int]
        lib.ocrt_rand_seed.argtypes = [C.POINTER(_ORand), C.c_uint]
        lib.ocrt_rand_next.argtypes = [C.POINTER(_ORand)]
        lib.ocrt_rand_next.restype = C.c_int
        lib.ocrt_sincos14.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int]
        lib.ocrt_bpp.argtypes = [C.c_int]
        lib.ocrt_bpp.restype = C.c_int
        lib.ocrt_lcg_jump.argtypes = [C.c_uint, C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
        _oracle = lib
    return _oracle


class OracleEngine:
    """Same call sequence, on the CPU restatement."""

    def __init__(self, variant, outw, outh, fmt=layout.PIX_BGRA, out=None, seed=1):
        self.spec = layout.system_spec(variant)
        self.lib = oracle_lib()
        taps = layout.conv_taps(variant)
        if variant.endswith("_bloom"):
            self.sys = self.lib.ocrt_system_bloom(self.spec.system, self.spec.pattern)
        else:
            self.sys = (self.lib.ocrt_system_conv_taps(self.spec.system, self.spec.pattern, taps) if taps
                        else self.lib.ocrt_system(self.spec.system, self.spec.pattern))
        assert self.sys, "unknown system"
        self.mon = _OMonitor()
        bpp = max(1, layout.bpp4fmt(fmt))
        self.out = out if out is not None else np.zeros((outh, outw, bpp), dtype=np.uint8)
        assert self.lib.ocrt_monitor_create(self.sys, C.byref(self.mon), outw, outh, fmt,
                                            self.out.ctypes.data)
        self.rand = _ORand()
        self.lib.ocrt_rand_seed(C.byref(self.rand), seed)
        self.rgb = _ORgb()
        self.nes = _ONes()
        self.nesrgb = _ONesRgb()
        self._img = None

    def __del__(self):
        try:
            self.lib.ocrt_monitor_destroy(C.byref(self.mon))
        except Exception:
            pass

    def set(self, **kw):
        for k, v in kw.items():
            setattr(self.mon, k, v)
        return self

    def resize(self, outw, outh, fmt, out):
        self.out = out
        self.mon.outw, self.mon.outh, self.mon.out_format = outw, outh, fmt
        self.mon.out = out.ctypes.data

    def reset(self):
        self.lib.ocrt_monitor_reset(C.byref(self.mon))

    def modulate(self, img, **kw):
        self._img = np.ascontiguousarray(img)
        if self.spec.system == layout.SYS_NES:
            s = self.nes
            kw.pop("border_color", None)
        elif self.spec.system == layout.SYS_NESRGB:
            s = self.nesrgb
        else:
            s = self.rgb
            kw.pop("iirs_initialized", None)
        s.data = self._img.ctypes.data
        s.h, s.w = self._img.shape[0], self._img.shape[1]
        for k, v in kw.items():
            setattr(s, k, v)
        if self.spec.system == layout.SYS_NES:
            self.lib.ocrt_encode_nes(self.sys, C.byref(self.mon), C.byref(s))
        elif self.spec.system == layout.SYS_SNES:
            self.lib.ocrt_encode_snes(self.sys, C.byref(self.mon), C.byref(s))
        elif self.spec.system == layout.SYS_NESRGB:
            self.lib.ocrt_encode_nesrgb(self.sys, C.byref(self.mon), C.byref(s))
        elif self.spec.system == layout.SYS_TEMP:
            self.lib.ocrt_encode_template(self.sys, C.byref(self.mon), C.byref(s))
        elif self.spec.system == layout.SYS_PV1K:
            self.lib.ocrt_encode_pv1k(self.sys, C.byref(self.mon), C.byref(s))
        else:
            self.lib.ocrt_encode_rgb(self.sys, C.byref(self.mon), C.byref(s), C.byref(self.rand))

    def demodulate(self, noise=0):
        self.lib.ocrt_decode(self.sys, C.byref(self.mon), noise, C.byref(self.rand))

    # staged decode, for comparing the kernels' intermediate tables
    def noise_pass(self, noise=0):
        self.lib.ocrt_noise_pass(self.sys, C.byref(self.mon), noise, C.byref(self.rand))

    def sync_pass(self):
        table = (OLine * self.spec.lines)()
        field = self.lib.ocrt_sync_pass(self.sys, C.byref(self.mon), table)
        return field, table

    def line_pass(self, table, first=0, count=None):
        self.lib.ocrt_line_pass(self.sys, C.byref(self.mon), table, first,
                                self.spec.lines if count is None else count)

    @property
    def analog(self):
        return np.ctypeslib.as_array(self.mon.analog, shape=(self.spec.input_size,)).astype(np.int8).copy()

    @property
    def inp(self):
        return np.ctypeslib.as_array(self.mon.inp, shape=(self.spec.input_size,)).astype(np.int8).copy()

    @property
    def ccf(self):
        return np.array([[self.mon.ccf[n][x] for x in range(self.spec.cc_samples)] for n in range(self.spec.vper)])

    @property
    def hsync(self):
        return self.mon.hsync

    @property
    def vsync(self):
        return self.mon.vsync

    @property
    def rn(self):
        return self.mon.rn

    def state(self):
        return dict(analog=self.analog, inp=self.inp, out=self.out.copy(), ccf=self.ccf,
                    hsync=self.hsync, vsync=self.vsync, rn=self.rn)


def assert_same_state(a, b, what=""):
    """Bit-exact comparison of two engine states with a useful first-mismatch report.  A state of the reference is
    also recorded (or, replayed, compared through its recorded digest: see ref_result)."""
    for ours, ref in ((a, b), (b, a)):
        if isinstance(ref, RefState):
            want = ref_result(lambda: state_digest(ref), live=not ref.replayed)
            if ref.replayed:
                bad = [k for k, x, y in zip(STATE_KEYS, state_digest(ours), want) if x != y]
                assert not bad, "%s: %s differ from the reference's recorded state" % (what, ", ".join(bad))
                return
            break
    for key in ("hsync", "vsync", "rn"):
        assert a[key] == b[key], "%s %s: %r != %r" % (what, key, a[key], b[key])
    assert np.array_equal(a["ccf"], b["ccf"]), "%s ccf: %r != %r" % (what, a["ccf"], b["ccf"])
    for key in ("analog", "inp", "out"):
        x, y = a[key], b[key]
        assert x.shape == y.shape, "%s %s shape %r != %r" % (what, key, x.shape, y.shape)
        if not np.array_equal(x, y):
            bad = np.argwhere(x != y)
            first = tuple(int(v) for v in bad[0])
            raise AssertionError("%s %s: %d mismatches, first at %r: %r != %r" % (
                what, key, len(bad), first, x[first], y[first]))


def cli_sequence(engine, img, noise=0, progressive=False, field=0, **settings):
    """The accumulate loop of the CLI driver (crt_main.c:221-255)."""
    engine.set(blend=1, scanlines=1)
    s = dict(settings)
    s.setdefault("as_color", 1)
    f, fr = field & 1, 0
    for it in range(4):
        engine.modulate(img, field=f, frame=fr, **s)
        engine.demodulate(noise)
        if not progressive:
            f ^= 1
            engine.modulate(img, field=f, frame=fr, **s)
            engine.demodulate(noise)
            if (it & 1) == 0:
                fr ^= 1


class ProductEngine(CEngine):
    """The CUDA product library through the reference's own C interface (host buffers)."""

    def __init__(self, variant, outw, outh, fmt=layout.PIX_BGRA, out=None):
        from ntsc_crt_b200 import capi
        capi.load(variant)  # raises if the library is not built: there is no fallback
        super().__init__(capi.lib_path(variant), variant, outw, outh, fmt, out)


def diff_report(name, x, y, shape_hint=None):
    """One-line description of how two arrays differ (for the GPU diagnostics)."""
    x = np.asarray(x)
    y = np.asarray(y)
    if x.shape != y.shape:
        return "%s: SHAPE %r vs %r" % (name, x.shape, y.shape)
    bad = np.argwhere(x != y)
    if len(bad) == 0:
        return "%s: identical (%d values)" % (name, x.size)
    first = tuple(int(v) for v in bad[0])
    last = tuple(int(v) for v in bad[-1])
    return "%s: %d/%d differ, first %r got %r want %r, last %r" % (
        name, len(bad), x.size, first, x[first], y[first], last)
