"""The segmented search (seg_kernels.cuh, fzb_search_segments) replayed on the CPU emulator of tests/emu, as
test_emu_kernels.py does for the other suites: the bodies of tests/test_gpu_segments.py at sizes a CPU does in
seconds, so `pytest -m "not gpu"` covers the new kernels and their host code."""
import pytest

import conftest
import test_gpu_segments as T
from fuzzysearch_b200 import _native, search


@pytest.fixture(scope="module")
def emu_lib():
    return conftest.load_emulated_library()


@pytest.fixture()
def emu_device(emu_lib, monkeypatch):
    monkeypatch.setattr(_native, "_lib", emu_lib)
    monkeypatch.setenv("FZB_EMU_SMS", "2")
    saved = dict(search._WORKSPACE)
    search._WORKSPACE.clear()
    yield 0
    search.release_workspace()
    import gc
    gc.collect()
    search._WORKSPACE.update(saved)


@pytest.mark.parametrize("route", [r[0] for r in T.ROUTES])
def test_emu_segments_per_route(emu_device, route):
    for alphabet in ("dna", "ascii"):
        # the segments on both sides of the short-segment bound only for one alphabet (the LP routes are slow here)
        T.test_segments_match_oracle_per_route(emu_device, route, alphabet, long=alphabet == "dna")


def test_emu_segments_isolation_and_refusals(emu_device):
    T.test_segments_are_isolated(emu_device)
    T.test_refusals(emu_device)


def test_emu_segments_public_api(emu_device):
    T.test_public_api_matches_the_per_item_loop(emu_device)


def test_emu_segments_reference_records(emu_device):
    assert T.replay_golden(T.load_golden("ref_fuzz.json"), stride=7) > 150
    T.test_reference_short_reads_fixture(emu_device, stride=3)


def test_emu_segments_launch_count(emu_device):
    T.test_launch_count_does_not_grow_with_the_number_of_segments(emu_device, many=2000)
