import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import pkgload  # noqa: E402

pkgload.load()


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_runtest_setup(item):
    import support
    support.begin_test(item)  # the reference results a test compares with are counted per run of it


def pytest_runtest_teardown(item, nextitem):
    import support
    support.end_test()


def _cuda_ok():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


# Library variants written after the round's GPU budget was spent (checked through tests/simt/ only): their GPU
# tests run after everything that has already been green on a B200, so that with `-x` a first-contact failure there
# cannot hide the state of the verified variants.  Remove a name once its tests have passed on the GPU.
NOT_YET_RUN_ON_GPU = ("template", "pv1k", "nes_p1", "nesrgb_p", "bloom", "test_gpu_wire", "test_gpu_still_cli", "test_gpu_edges", "test_gpu_fullsize", "newer_variants", "other_systems", "test_gpu_batch_api")


def pytest_collection_modifyitems(config, items):
    late = [it for it in items if "gpu" in it.keywords and any(n in it.nodeid for n in NOT_YET_RUN_ON_GPU)]
    if late:
        ids = set(id(it) for it in late)
        items[:] = [it for it in items if id(it) not in ids] + late
    if _cuda_ok():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)
