"""The minimal boundary types in pyscenedetect_b200/compat.py (used when the real `scenedetect`
package is not importable, e.g. on the GPU box) behave like the reference's classes for the
constant-frame-rate, frame-number-backed cases the hot path produces.  The reference's behaviour on
the same seeded sequences is stored in tests/golden/reference_boundary.json
(tests/golden/make_reference_boundary.py)."""

import json

import pytest

import pyscenedetect_b200.compat as compat_mod
from tests import reference_boundary as B


@pytest.fixture(scope="module")
def ref():
    with open(B.BOUNDARY_PATH) as f:
        return json.load(f)["compat"]


@pytest.fixture(scope="module")
def ours():
    c = compat_mod
    if c.USING_REFERENCE:
        pytest.skip("compat is already delegating to the reference")
    return c


@pytest.mark.parametrize("fps", B.FPS_CASES)
def test_frame_timecode_semantics(ref, ours, fps):
    want = ref["frame_timecode"][repr(fps)]
    got = B.frame_timecode_obs(ours.FrameTimecode, fps)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, (i, g, w)


@pytest.mark.parametrize("mode", B.FLASH_MODES)
@pytest.mark.parametrize("length", B.FLASH_LENGTHS)
def test_flash_filter_sequences(ref, ours, mode, length):
    want = ref["flash_filter"][f"{mode}/{length!r}"]
    assert B.flash_filter_obs(ours.FrameTimecode, ours.FlashFilter, mode, length) == want


def test_stats_manager_csv(ref, ours):
    got = B.stats_manager_obs(ours.FrameTimecode, ours.StatsManager)
    assert got[:2] == [True, False]
    assert got == ref["stats_manager"]
