"""The reference-side types at the plug-in boundary.

When the real `scenedetect` package is importable, its own `SceneDetector`, `FlashFilter`,
`FrameTimecode` and `StatsManager` are used unchanged (scenedetect/detector.py:37-224,
common.py:191-811, stats_manager.py:85-314) - the detectors in this package then subclass the
reference's ABC and drop straight into the reference `SceneManager`.

Where `scenedetect` is not importable, the minimal, independently written equivalents below
are used instead.  They implement only the constant-frame-rate, frame-number-backed behaviour
the hot path needs, with the same observable semantics (comparison/rounding rules, CSV layout),
and are pinned against the real classes' recorded behaviour by tests/test_compat_vs_reference.py.
"""

from __future__ import annotations

import csv
import math
import os
from abc import ABC, abstractmethod
from enum import Enum
from fractions import Fraction

USING_REFERENCE = False
if os.environ.get("PSD_B200_FORCE_COMPAT", "") != "1":
    try:  # pragma: no cover - depends on the environment
        from scenedetect.common import FrameTimecode  # type: ignore
        from scenedetect.detector import FlashFilter, SceneDetector  # type: ignore
        from scenedetect.stats_manager import StatsManager  # type: ignore

        USING_REFERENCE = True
    except Exception:  # ImportError or a broken partial install
        USING_REFERENCE = False


def _to_fraction(fps) -> Fraction:
    if isinstance(fps, Fraction):
        return fps
    if isinstance(fps, int):
        return Fraction(fps, 1)
    if hasattr(fps, "frame_rate") and not isinstance(fps, (int, float)):
        return fps.frame_rate
    fps = float(fps)
    for num in (24000, 30000, 60000, 120000):  # NTSC-like rates -> x/1001
        if abs(fps - num / 1001.0) < 1e-3:
            return Fraction(num, 1001)
    return Fraction(fps).limit_denominator(1000000)


if not USING_REFERENCE:

    def _parse_seconds(text: str, rate: Fraction) -> float:
        text = text.strip()
        if text.isdigit():
            return int(text) / float(rate)
        if ":" in text:
            parts = text.split(":")
            if len(parts) not in (2, 3):
                raise ValueError("Invalid timecode (too many separators).")
            nums = [float(p) if "." in p else int(p) for p in parts]
            if len(nums) == 2:
                nums = [0, *nums]
            hrs, mins, secs = nums
            if not (hrs >= 0 and 0 <= mins < 60 and 0 <= secs < 60):
                raise ValueError("Invalid timecode range (values outside allowed range).")
            return secs + hrs * 3600 + mins * 60
        if text.endswith("s"):
            text = text[:-1]
        if not text.replace(".", "").isdigit():
            raise ValueError("All characters in timecode seconds string must be digits.")
        return float(text)

    class FrameTimecode:
        """Frame position at a constant frame rate.  Either an exact frame number (what a
        `VideoStream.position` yields) or a number of seconds (float / string inputs)."""

        __slots__ = ("_frames", "_secs", "_rate")

        def __init__(self, timecode, fps=None):
            if isinstance(timecode, FrameTimecode):
                self._frames, self._secs = timecode._frames, timecode._secs
                self._rate = timecode._rate if fps is None else _to_fraction(fps)
                return
            if fps is None:
                raise TypeError("fps is a required argument.")
            self._rate = _to_fraction(fps)
            if self._rate <= 0:
                raise ValueError("Framerate must be positive and greater than zero.")
            self._frames, self._secs = None, None
            if isinstance(timecode, str) and timecode.isdigit():
                timecode = int(timecode)
            if isinstance(timecode, str):
                self._secs = _parse_seconds(timecode, self._rate)
            elif isinstance(timecode, float):
                if timecode < 0.0:
                    raise ValueError("Timecode frame number must be positive and greater than zero.")
                self._secs = timecode
            elif isinstance(timecode, int):
                if timecode < 0:
                    raise ValueError("Timecode frame number must be positive and greater than zero.")
                self._frames = timecode
            else:
                raise TypeError("Timecode format/type unrecognized.")

        @property
        def frame_rate(self) -> Fraction:
            return self._rate

        @property
        def framerate(self) -> float:
            return float(self._rate)

        @property
        def frame_num(self) -> int:
            if self._frames is not None:
                return self._frames
            return round(self._secs * self._rate)

        @property
        def seconds(self) -> float:
            if self._secs is not None:
                return self._secs
            return float(self._frames / self._rate)

        def get_frames(self) -> int:
            return self.frame_num

        def get_timecode(self, precision: int = 3, use_rounding: bool = True) -> str:
            secs = self.frame_num / float(self._rate)
            hrs = int(secs / 3600.0)
            secs -= hrs * 3600.0
            mins = int(secs / 60.0)
            secs = max(0.0, secs - mins * 60.0)
            if use_rounding:
                secs = round(secs, precision)
            secs = min(60.0, secs)
            if int(secs) == 60:
                secs, mins = 0.0, mins + 1
                if mins >= 60:
                    mins, hrs = 0, hrs + 1
            msec = format(secs, f".{precision + 1}f") if precision else ""
            return f"{hrs:02d}:{mins:02d}:{int(secs):02d}{msec[-(2 + precision):-1]}"

        # -- comparisons: ints compare frame numbers; floats/strings are converted to frames
        #    with round(seconds * rate) unless this object itself is seconds-backed --
        def _other_frames(self, other) -> int:
            if isinstance(other, int):
                return other
            if isinstance(other, float):
                return round(other * self._rate)
            if isinstance(other, str):
                return round(_parse_seconds(other, self._rate) * self._rate)
            if isinstance(other, FrameTimecode):
                if other._rate != self._rate:
                    raise ValueError(
                        "FrameTimecode instances require equal frame rate for frame-based arithmetic.")
                return other.frame_num
            raise TypeError("Unsupported type for performing arithmetic with FrameTimecode.")

        def _other_seconds(self, other) -> float:
            if isinstance(other, int):
                return float(other) / float(self._rate)
            if isinstance(other, float):
                return other
            if isinstance(other, str):
                return _parse_seconds(other, self._rate)
            if isinstance(other, FrameTimecode):
                return other.seconds
            raise TypeError("Unsupported type for performing arithmetic with FrameTimecode.")

        def _cmp(self, other, op) -> bool:
            if isinstance(other, int) or self._secs is None:
                return op(self.frame_num, self._other_frames(other))
            return op(self.seconds, self._other_seconds(other))

        def __eq__(self, other):
            if other is None:
                return False
            return self._cmp(other, lambda a, b: a == b)

        def __ne__(self, other):
            return not self.__eq__(other)

        def __lt__(self, other):
            return self._cmp(other, lambda a, b: a < b)

        def __le__(self, other):
            return self._cmp(other, lambda a, b: a <= b)

        def __gt__(self, other):
            return self._cmp(other, lambda a, b: a > b)

        def __ge__(self, other):
            return self._cmp(other, lambda a, b: a >= b)

        def __sub__(self, other):
            out = FrameTimecode(self)
            if self._secs is not None:
                out._secs = max(0.0, self._secs - self._other_seconds(other))
            else:
                out._frames = max(0, self._frames - self._other_frames(other))
            return out

        def __add__(self, other):
            out = FrameTimecode(self)
            if self._secs is not None:
                out._secs = self._secs + self._other_seconds(other)
            else:
                out._frames = self._frames + self._other_frames(other)
            return out

        def __int__(self):
            return self.frame_num

        def __float__(self):
            return self.seconds

        def __hash__(self):
            return self.frame_num

        def __str__(self):
            return self.get_timecode()

        def __repr__(self):
            return f"{self.get_timecode()} [frame_num={self.frame_num}, fps={self._rate}]"

    class StatsManager:
        """Per-frame metric store keyed by FrameTimecode, with the reference CSV layout:
        `Frame Number,Timecode,<sorted metric keys>`; row = frame_num+1, HH:MM:SS.nnn, str(v)."""

        def __init__(self, base_timecode=None):
            self._frame_metrics: dict = {}
            self._metric_keys: set[str] = set()
            self._metrics_updated = False
            self._base_timecode = base_timecode

        @property
        def metric_keys(self):
            return self._metric_keys

        def register_metrics(self, metric_keys) -> None:
            self._metric_keys = self._metric_keys.union(set(metric_keys))

        def get_metrics(self, timecode, metric_keys) -> list:
            row = self._frame_metrics.get(timecode, {})
            return [row.get(k) for k in metric_keys]

        def set_metrics(self, timecode, metric_kv_dict) -> None:
            self._metrics_updated = True
            self._frame_metrics.setdefault(timecode, {}).update(metric_kv_dict)

        def metrics_exist(self, timecode, metric_keys) -> bool:
            row = self._frame_metrics.get(timecode)
            return row is not None and all(k in row for k in metric_keys)

        def is_save_required(self) -> bool:
            return self._metrics_updated

        def save_to_csv(self, csv_file, force_save=True) -> None:
            if not (force_save or self.is_save_required()):
                return
            if isinstance(csv_file, (str, bytes, os.PathLike)):
                with open(csv_file, "w") as f:
                    self.save_to_csv(f, force_save)
                return
            writer = csv.writer(csv_file, lineterminator="\n")
            keys = sorted(self._metric_keys)
            writer.writerow(["Frame Number", "Timecode", *keys])
            for tc in sorted(self._frame_metrics.keys()):
                if not isinstance(tc, FrameTimecode):
                    continue
                writer.writerow([tc.frame_num + 1, tc.get_timecode()]
                                + [str(v) for v in self.get_metrics(tc, keys)])

    class SceneDetector(ABC):
        """The plug-in interface SceneManager drives (one call per frame)."""

        def __init__(self):
            self._stats_manager = None

        @abstractmethod
        def process_frame(self, timecode, frame_img) -> list:
            """Return the cuts detected with this frame (possibly earlier than `timecode`)."""

        def post_process(self, timecode) -> list:
            return []

        @property
        def event_buffer_length(self) -> int:
            return 0

        @property
        def stats_manager(self):
            return self._stats_manager

        @stats_manager.setter
        def stats_manager(self, value):
            self._stats_manager = value

        def get_metrics(self) -> list[str]:
            return []

    class FlashFilter:
        """Minimum-scene-length filter over the `score >= threshold` flag stream."""

        class Mode(Enum):
            MERGE = 0
            SUPPRESS = 1

        def __init__(self, mode, length):
            self._mode = mode
            self._filter_length = 0
            self._filter_secs = None
            if isinstance(length, float):
                self._filter_secs = length
            elif isinstance(length, str) and not length.strip().isdigit():
                self._filter_secs = FrameTimecode(timecode=length, fps=100.0).seconds
            elif isinstance(length, FrameTimecode):
                self._filter_secs = length.seconds
            else:
                self._filter_length = int(length)
            self._last_above = None
            self._merge_enabled = False
            self._merge_triggered = False
            self._merge_start = None

        @property
        def max_behind(self) -> int:
            if self._mode == FlashFilter.Mode.SUPPRESS:
                return 0
            if self._filter_secs is not None:
                return math.ceil(self._filter_secs * 240.0)
            return self._filter_length

        @property
        def _is_disabled(self) -> bool:
            if self._filter_secs is not None:
                return self._filter_secs <= 0.0
            return self._filter_length <= 0

        def filter(self, timecode, above_threshold: bool) -> list:
            if self._is_disabled:
                return [timecode] if above_threshold else []
            if self._last_above is None:
                self._last_above = timecode
            if self._filter_secs is None:  # fixed once from the first frame's rate
                self._filter_secs = self._filter_length / float(timecode.frame_rate)
            met = (timecode - self._last_above) >= self._filter_secs
            if self._mode == FlashFilter.Mode.SUPPRESS:
                if not (above_threshold and met):
                    return []
                self._last_above = timecode
                return [timecode]
            if self._mode != FlashFilter.Mode.MERGE:
                raise RuntimeError("Unhandled FlashFilter mode.")
            if above_threshold:
                self._last_above = timecode
            if self._merge_triggered:
                if (met and not above_threshold
                        and (self._last_above - self._merge_start) >= self._filter_secs):
                    self._merge_triggered = False
                    return [self._last_above]
                return []
            if not above_threshold:
                return []
            if met:
                self._merge_enabled = True
                return [timecode]
            if self._merge_enabled:
                self._merge_triggered = True
                self._merge_start = timecode
            return []


__all__ = ["FrameTimecode", "StatsManager", "SceneDetector", "FlashFilter", "USING_REFERENCE"]
