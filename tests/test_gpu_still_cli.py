"""tools/crtx_still.c, the batch counterpart of the reference's command-line driver: for every (in, out) pair the file
it writes must be byte-identical to what the all-reference build of crt_main.c (oracle/_ref/cli_ref_ntsc) writes for
that pair alone -- PPM and BMP, in and out, every flag of the command line, several images in one run.  Where that build
is absent, the reference's files are known by the length and digest recorded under tests/golden/reference/."""
import os
import struct
import subprocess

import numpy as np
import pytest

import support as S

pytestmark = pytest.mark.gpu

REF_CLI = os.path.join(S.REF_DIR, "cli_ref_ntsc")
STILL = os.path.join(S.ROOT, "ntsc-crt_b200", "bin", "crtx_still")


def write_ppm(path, rgb, maxc=255, comment=False):
    with open(path, "wb") as f:
        f.write(b"P6\n" + (b"# made by a test\n" if comment else b"") + b"%d %d\n%d\n" % (rgb.shape[1], rgb.shape[0], maxc))
        f.write(rgb.tobytes())


def write_bmp(path, bgra, bits):
    h, w = bgra.shape[:2]
    bpp = bits // 8
    pad = (4 - (w * bpp) % 4) % 4
    rows = b"".join(bgra[y, :, :bpp].tobytes() + b"\0" * pad for y in range(h - 1, -1, -1))
    head = b"BM" + struct.pack("<IHHI", 54 + len(rows), 0, 0, 54) + struct.pack("<IiiHHIIiiII", 40, w, h, 1, bits, 0, len(rows), 0, 0, 0, 0)
    with open(path, "wb") as f:
        f.write(head + rows)


@pytest.mark.skipif(not os.path.exists(STILL), reason="driver not built")
@pytest.mark.parametrize("flags,outw,outh,noise,hue", [("-o", 832, 624, 0, 0), ("-op", 640, 480, 12, 30), ("-omf", 333, 250, 24, 0),
                                                       ("-opr", 832, 624, 0, 90), ("-opa", 320, 240, 0, 0)])
def test_batch_still_driver_is_byte_identical_to_the_reference_cli(tmp_path, flags, outw, outh, noise, hue):
    rng = np.random.default_rng(outw + noise)
    inputs = []
    a = S.bars_image(320, 240, fmt=S.layout.PIX_RGB)[..., :3].copy()
    write_ppm(str(tmp_path / "a.ppm"), a)
    inputs.append(("a.ppm", "a_out.ppm"))
    b = rng.integers(0, 256, size=(200, 301, 3), dtype=np.uint8)  # odd width, comment line in the header
    write_ppm(str(tmp_path / "b.ppm"), b, comment=True)
    inputs.append(("b.ppm", "b_out.bmp"))
    c = rng.integers(0, 101, size=(64, 48, 3), dtype=np.uint8)  # maximum colour value 100: rescaled (ppm_rw.c:80)
    write_ppm(str(tmp_path / "c.ppm"), c, maxc=100)
    inputs.append(("c.ppm", "c_out.ppm"))
    d = S.rand_image(257, 199, seed=4)
    write_bmp(str(tmp_path / "d.bmp"), d, 24)
    inputs.append(("d.bmp", "d_out.bmp"))
    e = S.rand_image(640, 480, seed=5)
    write_bmp(str(tmp_path / "e.bmp"), e, 32)
    inputs.append(("e.bmp", "e_out.ppm"))
    args = []
    for i, o in inputs:
        args += [i, o]
    res = subprocess.run([STILL, flags, str(outw), str(outh), str(noise), str(hue)] + args, cwd=str(tmp_path),
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert res.returncode == 0, res.stderr.decode() + res.stdout.decode()
    for i, o in inputs:
        def ref_file():
            want = str(tmp_path / ("ref_" + o))
            subprocess.run([REF_CLI, flags if "o" in flags else flags + "o", str(outw), str(outh), str(noise), str(hue), i, want],
                           cwd=str(tmp_path), check=True, stdout=subprocess.DEVNULL, timeout=300)
            ref = open(want, "rb").read()
            return [len(ref), S.digest(np.frombuffer(ref, dtype=np.uint8))]
        got = open(tmp_path / o, "rb").read()
        ref_len, ref_digest = S.ref_result(ref_file, os.path.exists(REF_CLI))
        assert ref_len > 1000
        assert [len(got), S.digest(np.frombuffer(got, dtype=np.uint8))] == [ref_len, ref_digest], (
            "%s -> %s differs from the reference CLI's file (flags %s)" % (i, o, flags))


def test_usage_errors():
    if not os.path.exists(STILL):
        pytest.skip("driver not built")
    assert subprocess.run([STILL], stdout=subprocess.DEVNULL).returncode != 0
    assert subprocess.run([STILL, "-o", "832", "624", "0", "0", "only_one_file"], stdout=subprocess.DEVNULL).returncode != 0
    assert subprocess.run([STILL, "-z", "832", "624", "0", "0", "a", "b"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL).returncode != 0
