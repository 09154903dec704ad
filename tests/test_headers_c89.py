"""The public headers are what the reference's C89 drivers and tools/crtx_video.c include: they must compile as
strict C89 for every system the library ships, and lay `struct CRT` / `struct NTSC_SETTINGS` out exactly as the
compiled reference does (sizes probed from oracle/_ref, else recorded under tests/golden/reference/)."""
import ctypes as C
import os
import subprocess
import tempfile

import pytest

import support as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INC = os.path.join(ROOT, "include")

SYSTEMS = [("ntsc", ["-DCRT_SYSTEM=0"]), ("vhs", ["-DCRT_SYSTEM=5"]), ("nes", ["-DCRT_SYSTEM=1"]),
           ("nes_p0", ["-DCRT_SYSTEM=1", "-DCRT_CHROMA_PATTERN=0"]), ("nes_p1", ["-DCRT_SYSTEM=1", "-DCRT_CHROMA_PATTERN=1"]), ("snes", ["-DCRT_SYSTEM=3"]),
           ("nesrgb", ["-DCRT_SYSTEM=6"]), ("nesrgb_p0", ["-DCRT_SYSTEM=6", "-DCRT_CHROMA_PATTERN=0"]),
           ("nesrgb_p1", ["-DCRT_SYSTEM=6", "-DCRT_CHROMA_PATTERN=1"]), ("template", ["-DCRT_SYSTEM=4"]), ("pv1k", ["-DCRT_SYSTEM=2"])]

PROBE = r"""
#include <stdio.h>
#include "crt_core.h"      /* the compat shim: resolves to crt_b200.h */
#include "crtx_batch.h"
int main(void)
{
    printf("%d %d %d %d %d\n", (int) sizeof(struct CRT), (int) sizeof(struct NTSC_SETTINGS), CRT_HRES, CRT_INPUT_SIZE,
           CRT_CC_VPER);
    return 0;
}
"""


@pytest.mark.parametrize("variant,defs", SYSTEMS)
def test_headers_compile_as_c89_and_match_the_reference_layout(variant, defs):
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "probe.c")
        exe = os.path.join(tmp, "probe")
        with open(src, "w") as f:
            f.write(PROBE)
        cmd = ["gcc", "-std=c89", "-pedantic", "-Wall", "-Werror", "-I" + os.path.join(INC, "compat"), "-I" + INC] + defs + [src, "-o", exe]
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        assert res.returncode == 0, res.stderr.decode()
        out = subprocess.run([exe], stdout=subprocess.PIPE, check=True).stdout.split()
    size_crt, size_set, hres, input_size, vper = (int(x) for x in out)
    spec = S.layout.system_spec(variant)
    assert (hres, input_size, vper) == (spec.hres, spec.input_size, spec.vper)
    assert size_crt == C.sizeof(S.layout.crt_struct(spec))
    assert size_set == C.sizeof(S.layout.settings_struct(spec))
    def ref_sizes():
        lib = C.CDLL(S.ref_path(variant))
        return [lib.ref_sizeof_crt(), lib.ref_sizeof_settings()]
    assert [size_crt, size_set] == S.ref_result(ref_sizes, S.have_ref(variant))


@pytest.mark.parametrize("prog", ["crtx_video", "crtx_still"])
def test_batch_drivers_are_strict_c89(prog):
    """tools/crtx_video.c and tools/crtx_still.c must build with -std=c89 -pedantic -Werror against crtx_batch.h alone
    (no CUDA header)."""
    with tempfile.TemporaryDirectory() as tmp:
        cmd = ["gcc", "-std=c89", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I" + INC, "-c",
               os.path.join(ROOT, "tools", prog + ".c"), "-o", os.path.join(tmp, prog + ".o")]
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        assert res.returncode == 0, res.stderr.decode()
