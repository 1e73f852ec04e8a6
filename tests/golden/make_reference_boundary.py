#!/usr/bin/env python
"""Generate tests/golden/reference_boundary.json from a PySceneDetect 0.7.1 source checkout:

    python tests/golden/make_reference_boundary.py PATH/TO/PySceneDetect

Records, with the reference's own classes:
  * `compat`: FrameTimecode, FlashFilter and StatsManager observations (tests/reference_boundary.py);
  * `scene_manager_traces`: for every golden case, the calls the reference `SceneManager.detect_scenes`
    makes on a detector - the frame number of every `process_frame`, a hash of the frames it passes
    (cropped / downscaled as the SceneManager does), `post_process`, and the start / last positions the
    scene list is built from;
  * `scene_manager_settings`: frames read, cut list and scene list of the reference SceneManager with
    the reference ContentDetector over end_time / duration / frame_skip / crop settings.
"""

from __future__ import annotations

import hashlib
import json
import os
import sys
from fractions import Fraction

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def main():
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "scenedetect")):
        raise SystemExit(__doc__)
    sys.path.insert(0, ROOT)
    sys.path.append(os.path.abspath(sys.argv[1]))  # after ROOT: the checkout has its own `tests` package

    import numpy as np
    import scenedetect
    from scenedetect.common import FrameTimecode
    from scenedetect.detector import FlashFilter, SceneDetector
    from scenedetect.detectors import ContentDetector
    from scenedetect.scene_manager import SceneManager
    from scenedetect.stats_manager import StatsManager
    from scenedetect.video_stream import VideoStream

    from tests import reference_boundary as B
    from tests.golden_util import case_frames, case_names, get_case

    class RefStream(B.SyntheticStream, VideoStream):
        pass

    class Spy(SceneDetector):
        def __init__(self, keys):
            super().__init__()
            self.keys, self.frames, self.post = keys, [], []
            self.sha, self.shape = hashlib.sha256(), None

        def get_metrics(self):
            return self.keys

        def process_frame(self, timecode, frame_img):
            self.frames.append(timecode.frame_num)
            self.sha.update(np.ascontiguousarray(frame_img).tobytes())
            self.shape = list(frame_img.shape)
            return []

        def post_process(self, timecode):
            self.post.append(timecode.frame_num)
            return []

    out = {"reference_version": scenedetect.__version__, "compat": {}, "scene_manager_traces": {},
           "scene_manager_settings": {}}
    c = out["compat"]
    c["frame_timecode"] = {repr(fps): B.frame_timecode_obs(FrameTimecode, fps) for fps in B.FPS_CASES}
    c["flash_filter"] = {f"{m}/{length!r}": B.flash_filter_obs(FrameTimecode, FlashFilter, m, length)
                         for m in B.FLASH_MODES for length in B.FLASH_LENGTHS}
    c["stats_manager"] = B.stats_manager_obs(FrameTimecode, StatsManager)

    for name in case_names():
        case = get_case(name)
        frames = case_frames(case)
        stats = StatsManager() if case["stats"] else None
        sm = SceneManager(stats)
        spy = Spy(case.get("metric_keys") or [])
        sm.add_detector(spy)
        if case["mode"] == "scene_manager" and case.get("auto_downscale"):
            sm.auto_downscale = True
        else:
            sm.auto_downscale = False
            sm.downscale = case.get("downscale", 1)
        stream = RefStream(frames, case["fps"], timecode=FrameTimecode)
        n = sm.detect_scenes(stream)
        assert spy.frames == list(range(spy.frames[0], spy.frames[0] + len(spy.frames)))
        out["scene_manager_traces"][name] = {
            "frames_read": n, "fps": str(Fraction(stream.frame_rate)),
            "first_frame": spy.frames[0], "frame_count": len(spy.frames),
            "frame_shape": spy.shape, "frames_sha256": spy.sha.hexdigest(), "post_process": spy.post,
            "start_pos": sm._start_pos.frame_num, "last_pos": sm._last_pos.frame_num,
            "stats_manager_bound": spy.stats_manager is stats}

    frames = case_frames(get_case("content_default_nostats"))
    for st in B.SM_SETTINGS:
        sm = SceneManager()
        sm.add_detector(ContentDetector())
        out["scene_manager_settings"][B.settings_key(st)] = B.run_scene_manager(
            sm, RefStream(frames, 30.0, timecode=FrameTimecode), st)

    with open(B.BOUNDARY_PATH, "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")
    print("wrote", B.BOUNDARY_PATH, os.path.getsize(B.BOUNDARY_PATH), "bytes")


if __name__ == "__main__":
    main()
