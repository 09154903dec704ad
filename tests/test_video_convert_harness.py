"""CPU half of tests/test_gpu_video_convert_unmodified.py: pins the stack-clearing harness (oracle/zero_stack_main.c) in
front of the reference's UNMODIFIED extra/video_convert.c against the oracle's sequential loop."""
import os

import numpy as np
import pytest

import support as S
from ntsc_crt_b200 import layout
from test_gpu_video_driver import moving_bars, read_bmp32
from test_gpu_video_convert_unmodified import REF_VIDEO, run_driver


@pytest.mark.parametrize("flags,noise", [("-o", 0), ("-om", 7)])
def test_reference_video_driver_with_a_cleared_stack_is_the_sequential_loop(tmp_path, flags, noise):
    """CPU only: pins the harness -- with the stack cleared the unmodified driver equals the oracle's loop with
    xoffset = yoffset = 0 (video_convert.c:226-277: blend 0, scanlines 1, field toggles every image, frame every other).
    Where the driver is not built, its images are the ones recorded under tests/golden/reference/."""
    frames = moving_bars(6, 320, 240, seed=2)

    def ref_images():
        files = run_driver(REF_VIDEO, str(tmp_path), frames, flags, 640, 480, noise)
        return [S.digest(read_bmp32(str(tmp_path / "output" / ("%06d.bmp" % (k + 1))))) for k in range(len(files))]
    live = os.path.exists(REF_VIDEO)
    want = S.ref_result(ref_images, live)
    ora = S.OracleEngine("ntsc", 640, 480)
    ora.set(blend=0, scanlines=1, saturation=10)
    field = frame = 0
    for k in range(len(frames)):
        ora.modulate(frames[k], format=layout.PIX_BGRA, as_color=0 if "m" in flags else 1, field=field, frame=frame, raw=0, hue=0)
        ora.demodulate(noise)
        field ^= 1
        if ((k + 1) & 1) == 0:
            frame ^= 1
        if live:
            got = read_bmp32(str(tmp_path / "output" / ("%06d.bmp" % (k + 1))))
            assert np.array_equal(got, ora.out), "image %d: %s" % (k + 1, S.diff_report("pixels", got, ora.out))
        assert S.digest(ora.out) == want[k], "image %d differs from the reference driver's" % (k + 1)
    assert len(want) == 6
