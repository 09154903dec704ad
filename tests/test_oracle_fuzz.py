"""The seeded random sweep of tests/test_gpu_fuzz.py, run on the CPU between the oracle and the COMPILED
REFERENCE (oracle/_ref, else its states recorded under tests/golden/reference/): it widens the pinning of the oracle beyond the hand-picked cases and proves that every
configuration the GPU sweep draws lies inside the reference's defined behaviour (so a GPU mismatch there is a bug,
never an artefact of undefined reads)."""
import importlib.util
import os

import numpy as np
import pytest

import support as S
from ntsc_crt_b200 import layout

_spec = importlib.util.spec_from_file_location("gpu_fuzz", os.path.join(os.path.dirname(os.path.abspath(__file__)), "test_gpu_fuzz.py"))
gpu_fuzz = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(gpu_fuzz)


@pytest.mark.parametrize("variant,seed", [("ntsc", 1), ("ntsc", 3), ("ntsc_conv", 4), ("nes", 6), ("nes_p0", 7),
                                          ("snes", 10), ("ntsc_conv5", 11), ("template", 12), ("pv1k", 13), ("ntsc_bloom", 14),
                                          ("pv1k", 15), ("template", 16), ("ntsc_bloom", 17)])
def test_gpu_sweep_cases_are_inside_the_reference_domain(variant, seed):
    rng = np.random.default_rng(1000 + seed)  # the same stream the GPU sweep consumes
    for case in range(4):
        fmt, outw, outh, knobs, w, h = gpu_fuzz.draw_case(rng, variant)
        ref = S.ref_engine(variant, outw, outh, fmt, seed=1)
        ora = S.OracleEngine(variant, outw, outh, fmt)
        for e in (ref, ora):
            e.set(**knobs)
        nes = variant.startswith("nes")
        if nes:
            img = rng.integers(0, 512, size=(h, w), dtype=np.uint16)
        else:
            src_fmt = int(rng.integers(0, 6))
            img = S.pack_rgb(S.rand_image(w, h, bpp=3, seed=int(rng.integers(0, 1 << 30))), src_fmt)
        for call in range(3):
            noise = int(rng.choice([0, 0, 3, 12, 40, 255]))
            if nes:
                kw = dict(dot_crawl_offset=int(rng.integers(0, 3)), hue=int(rng.integers(0, 360)),
                          xoffset=int(rng.integers(0, 3)) * 4, yoffset=int(rng.integers(0, 3)))
            else:
                field = int(rng.integers(0, 2))
                kw = dict(format=src_fmt, as_color=int(rng.integers(0, 2)), field=field, frame=int(rng.integers(0, 2)),
                          raw=0, hue=int(rng.integers(0, 360)), xoffset=int(rng.integers(0, 4)) * 4,
                          yoffset=int(rng.integers(0, 3)))
                if variant in ("snes", "template", "pv1k"):
                    kw["dot_crawl_offset"] = int(rng.integers(0, 4))
            for e in (ref, ora):
                e.modulate(img, **kw)
                e.demodulate(noise)
            S.assert_same_state(ref.state(), ora.state(), "%s seed %d case %d call %d" % (variant, seed, case, call))
