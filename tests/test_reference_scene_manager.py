"""Drop-in boundary, both directions, against what the reference's `SceneManager` does
(tests/golden/reference_boundary.json, recorded from PySceneDetect 0.7.1 by
tests/golden/make_reference_boundary.py):

  1. every golden case: this package's detector driven by the exact call sequence the reference's
     `SceneManager.detect_scenes` issues (frame numbers, frames as it crops / downscales them,
     `post_process`) - cut list, scene list and CSV hash must equal what the reference's CPU detector
     produced (tests/golden/golden_v1.json, golden_v2.json);
  2. this package's batched SceneManager against the reference SceneManager driving the reference's CPU
     ContentDetector over end_time / duration (frames, seconds, timecode string) / frame_skip / crop.

CPU box: oracle-backed fake engine; GPU box: the real engine."""

import hashlib
import io
import json
from fractions import Fraction

import numpy as np
import pytest

import pyscenedetect_b200.detectors._base as base_mod
import pyscenedetect_b200.scene_manager as sm_mod
from oracle import ref_detectors as R
from tests import reference_boundary as B
from tests.golden_util import case_frames, case_names, get_case
from tests.test_gpu_parity import _build


def _replay_case(name):
    """Part 1 for one golden case -> list of mismatches."""
    from pyscenedetect_b200 import FrameTimecode, StatsManager
    with open(B.BOUNDARY_PATH) as f:
        trace = json.load(f)["scene_manager_traces"][name]
    case = get_case(name)
    frames = case_frames(case)
    if case["mode"] == "scene_manager" and case.get("auto_downscale"):
        factor = R.compute_downscale_factor(max(frames.shape[2], frames.shape[1]))
    else:
        factor = case.get("downscale", 1)
    first, count = trace["first_frame"], trace["frame_count"]
    passed = [R.downscale_frame(frames[i], factor) for i in range(first, first + count)]
    sha = hashlib.sha256()
    for fr in passed:
        sha.update(np.ascontiguousarray(fr).tobytes())
    assert sha.hexdigest() == trace["frames_sha256"] and list(passed[-1].shape) == trace["frame_shape"], \
        "frames differ from the ones the reference SceneManager passed"

    # what SceneManager.add_detector does, then detect_scenes' calls
    fps = Fraction(trace["fps"])
    stats = StatsManager() if case["stats"] else None
    det = _build(case)
    det.stats_manager = stats
    assert trace["stats_manager_bound"]
    if stats is not None:
        stats.register_metrics(det.get_metrics())
    cuts = []
    for i, fr in enumerate(passed):
        cuts += det.process_frame(FrameTimecode(first + i, fps), fr)
    for t in trace["post_process"]:
        cuts += det.post_process(FrameTimecode(t, fps))
    det.close()

    failures = []
    cut_list = sorted(set(cuts))
    if trace["frames_read"] != frames.shape[0] or [c.frame_num for c in cut_list] != case["cuts"]:
        failures.append(f"cuts:{name}")
    if case["scene_list"] is not None:
        scenes = sm_mod.get_scenes_from_cuts(cut_list, FrameTimecode(trace["start_pos"], fps),
                                             FrameTimecode(trace["last_pos"] + 1, fps)) if cut_list else []
        if [[a.frame_num, b.frame_num] for a, b in sorted(scenes)] != case["scene_list"]:
            failures.append(f"scenes:{name}")
    if stats is not None and not any(k.startswith("hist_diff") for k in case["metric_keys"]):
        buf = io.StringIO()
        stats.save_to_csv(buf)
        if hashlib.sha256(buf.getvalue().encode()).hexdigest() != case["csv_sha256"]:
            failures.append(f"csv:{name}")
    return failures


def _run():
    from pyscenedetect_b200.detectors import ContentDetector
    from pyscenedetect_b200.scene_manager import SceneManager
    from pyscenedetect_b200.video import ArrayVideoStream
    with open(B.BOUNDARY_PATH) as f:
        want_settings = json.load(f)["scene_manager_settings"]
    failures, checked = [], 0
    # ---- 1. our detectors under the reference SceneManager's calls ----
    for name in case_names():
        failures += _replay_case(name)
        checked += 1
    # ---- 2. our SceneManager vs the reference SceneManager + reference CPU detector ----
    frames = case_frames(get_case("content_default_nostats"))
    for st in B.SM_SETTINGS:
        want = want_settings[B.settings_key(st)]
        sm = SceneManager(batch_size=16)
        sm.add_detector(ContentDetector())
        got = B.run_scene_manager(sm, B.SyntheticStream(frames, 30.0), st)  # no read_batch: frame by frame
        checked += 1
        if got != want:
            failures.append(f"settings:{st}: ref={want} ours={got}")
        # and the zero-copy (read_batch) path of our SceneManager where it applies
        if "crop" not in st and not st.get("frame_skip") and not st.get("start"):
            sm = SceneManager(batch_size=16)
            sm.add_detector(ContentDetector())
            got = B.run_scene_manager(sm, ArrayVideoStream(frames, 30.0), st)
            checked += 1
            if got != want:
                failures.append(f"zero-copy settings:{st}: ref={want} ours={got}")
    assert failures == [] and checked >= 40, (checked, failures)


def test_reference_scene_manager_drives_our_detectors_fake_engine(monkeypatch):
    from tests.fake_engine import OracleEngine

    class FakePinned:
        def __init__(self, nbytes):
            self.array = np.zeros(nbytes, np.uint8)

        def close(self):
            pass
    monkeypatch.setattr(base_mod, "Engine", OracleEngine)
    monkeypatch.setattr(sm_mod, "Engine", OracleEngine)
    monkeypatch.setattr(sm_mod, "PinnedBuffer", FakePinned)
    _run()


@pytest.mark.gpu
def test_reference_scene_manager_drives_our_detectors_real_engine():
    _run()
