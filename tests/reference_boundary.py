"""What the boundary types and the reference `SceneManager` do, as plain data.

`tests/golden/make_reference_boundary.py` runs these functions on the real PySceneDetect classes and
stores the results in `tests/golden/reference_boundary.json`; `tests/test_compat_vs_reference.py` and
`tests/test_reference_scene_manager.py` run them on this package's classes and compare.  The sequences
are seeded and every float is stored as `float.hex()`, so a comparison is exact."""

from __future__ import annotations

import io
import os
import random
import zlib
from fractions import Fraction

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
BOUNDARY_PATH = os.path.join(HERE, "golden", "reference_boundary.json")

FPS_CASES = [30.0, 25.0, 24000 / 1001, 29.97, 60.0]
FLASH_MODES = ["MERGE", "SUPPRESS"]
FLASH_LENGTHS = [15, 0, 1, 40, 0.5, "0.6s", "00:00:00.700", "20"]
_CMP_OTHERS = (15, 0.5, 0.6, "0.6s", "00:00:01.250", "12", 1.0 / 3.0)

# SceneManager.detect_scenes settings compared on the "content_default_nostats" golden case
SM_SETTINGS = [dict(), dict(end_time=100), dict(end_time=3.5), dict(end_time="00:00:05.100"), dict(duration=77),
               dict(duration=2.0), dict(duration="3s"), dict(end_time=0), dict(duration=0), dict(frame_skip=1),
               dict(frame_skip=3, end_time=120), dict(crop=(143, 10, 16, 81)), dict(crop=(0, 0, 40, 30), auto=True),
               dict(crop=(100, 50, 400, 300)), dict(start=40, duration=60), dict(start=40, end_time=90)]


def settings_key(st: dict) -> str:
    return repr(sorted(st.items()))


def _bits(values) -> str:
    return "".join("1" if v else "0" for v in values)


def frame_timecode_obs(FrameTimecode, fps) -> list:
    """Frame numbers, timecode strings, seconds, arithmetic, comparisons and hashes of seeded timecodes."""
    rng = random.Random(1)
    out = []
    for _ in range(300):
        a, b = rng.randrange(0, 200000), rng.randrange(0, 200000)
        x, y = FrameTimecode(a, fps), FrameTimecode(b, fps)
        d = x - y
        cmp = [v for other in _CMP_OTHERS for v in (d >= other, x < other)]
        out.append([x.frame_num, x.get_timecode(), float(x.seconds).hex(), str(Fraction(x.frame_rate)),
                    d.frame_num, (x + 7).frame_num, _bits(cmp + [x == y, x >= y]), hash(x)])
    out.append([str(FrameTimecode("00:01:02.500", fps)), FrameTimecode(1.5, fps).frame_num])
    return out


def flash_filter_obs(FrameTimecode, FlashFilter, mode: str, length) -> list:
    """max_behind and every emitted cut of a seeded above/below-threshold sequence at two frame rates."""
    rng = random.Random(zlib.crc32(f"{mode}/{length!r}".encode()))
    out = []
    for fps in (30.0, 24000 / 1001):
        f = FlashFilter(FlashFilter.Mode[mode], length)
        p = rng.choice([0.05, 0.2, 0.5])
        emitted = []
        for t in range(600):
            above = rng.random() < p
            cuts = [c.frame_num for c in f.filter(FrameTimecode(t, fps), above)]
            if cuts:
                emitted.append([t, cuts])
        out.append([f.max_behind, emitted])
    return out


def stats_manager_obs(FrameTimecode, StatsManager) -> list:
    """metrics_exist, get_metrics and the CSV text of a StatsManager filled with seeded rows."""
    sm = StatsManager()
    keys = ["content_val", "delta_hue", "adaptive_ratio (w=2)"]
    sm.register_metrics(keys)
    rng = random.Random(3)
    for t in range(1, 80):
        row = {"content_val": np.float64(rng.random() * 50), "delta_hue": np.float64(rng.random())}
        if t % 3:
            row["adaptive_ratio (w=2)"] = rng.random() * 4
        sm.set_metrics(FrameTimecode(t, 30.0), row)
    buf = io.StringIO()
    sm.save_to_csv(buf)
    got = sm.get_metrics(FrameTimecode(3, 30.0), keys)
    return [sm.metrics_exist(FrameTimecode(5, 30.0), ["content_val"]),
            sm.metrics_exist(FrameTimecode(0, 30.0), ["content_val"]),
            [None if v is None else float(v).hex() for v in got], buf.getvalue()]


class SyntheticStream:
    """Forward-only, frame-by-frame `VideoStream` over an in-memory array (no `read_batch`)."""

    BACKEND_NAME = "synthetic"

    def __init__(self, frames, fps=30.0, timecode=None):
        if timecode is None:
            from pyscenedetect_b200.compat import FrameTimecode as timecode
        self._tc = timecode
        self._frames, self._n = frames, 0
        self._fps = Fraction(fps).limit_denominator(1000000)

    path = property(lambda self: "synthetic")
    name = property(lambda self: "synthetic")
    is_seekable = property(lambda self: False)
    frame_rate = property(lambda self: self._fps)
    duration = property(lambda self: self._tc(len(self._frames), self._fps))
    frame_size = property(lambda self: (self._frames.shape[2], self._frames.shape[1]))
    aspect_ratio = property(lambda self: 1.0)
    frame_number = property(lambda self: self._n)
    position = property(lambda self: self._tc(max(0, self._n - 1), self._fps))
    position_ms = property(lambda self: 0.0 if self._n == 0 else 1000.0 * (self._n - 1) / float(self._fps))

    def read(self, decode=True):
        if self._n >= len(self._frames):
            return False
        self._n += 1
        return self._frames[self._n - 1] if decode else True

    def reset(self):
        self._n = 0

    def seek(self, target):
        raise NotImplementedError


def run_scene_manager(sm, stream, st: dict) -> list:
    """sm.detect_scenes with one of SM_SETTINGS -> [frames read, cut frames, [start, end] scene frames]."""
    sm.auto_downscale = bool(st.get("auto", False))
    if "crop" in st:
        sm.crop = st["crop"]
    for _ in range(st.get("start", 0)):
        stream.read(decode=False)
    kw = {k: v for k, v in st.items() if k in ("end_time", "duration", "frame_skip")}
    n = sm.detect_scenes(stream, **kw)
    return [n, [c.frame_num for c in sm.get_cut_list()], [[a.frame_num, b.frame_num] for a, b in sm.get_scene_list()]]
