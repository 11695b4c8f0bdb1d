"""Batched, device-resident detect -> track path over many video streams.

The reference processes one frame of one stream per call, on the CPU except for the two
TensorRT engines (``/root/reference/src/aicamera_tracker.py:169-240``).  Here a batch of
frames (one per stream) goes through K1-K12 without leaving the GPU and without a host
synchronisation: detections, crop counts and track tables stay in fixed-capacity device
buffers.  ``YOLODetector`` / ``DeepSORT`` (the reference-shaped facades) are thin single-stream
wrappers around ``BatchDetector`` / ``BatchTracker``.
"""
import ctypes as C
import math
from dataclasses import dataclass, fields, replace
from typing import FrozenSet, Optional, Sequence, Tuple, Union

import torch

from . import _lib, config
from .trt_engine import TRTEngine


def resolve_thresholds(conf_threshold, min_detection_confidence=None):
    """(NMS score threshold, minimum detection confidence) of a detector confidence threshold, as one reference process
    applies them: the engine's NMS keeps scores >= min(conf, YOLO_CONF_THRESHOLD) (yolo_detector.py:131 then drops those
    below conf), and DeepSORT drops those below its own minimum (deepsort_tracker.py:88-95), on the device one comparison
    whose default is therefore max(DEEPSORT_MIN_CONFIDENCE, conf)."""
    score = min(conf_threshold, config.YOLO_CONF_THRESHOLD)
    if min_detection_confidence is None:
        min_detection_confidence = max(config.DEEPSORT_MIN_CONFIDENCE, conf_threshold)
    return score, min_detection_confidence


@dataclass(frozen=True)
class StreamSettings:
    """One stream's detection and tracking settings: what a reference process takes as constructor arguments
    (``YOLODetector(conf_threshold, nms_threshold)``, ``DeepSORT(max_cosine_distance, max_iou_distance, max_age, n_init,
    min_detection_confidence)``) and the class names it tracks.  ``min_detection_confidence`` None resolves as
    ``resolve_thresholds`` does.  ``include_regions`` / ``exclude_regions``: where in its frame the stream tracks, polygons of
    3 to 32 integer frame-pixel (x, y) vertices, at most 8 in all; a detection is tracked when the bottom centre of its box
    is inside some include polygon (or there is none) and inside no exclude polygon (include/aicam.h,
    aicam_frame_table_set_regions)."""
    conf_threshold: float = config.YOLO_CONF_THRESHOLD
    nms_threshold: float = config.YOLO_NMS_THRESHOLD
    classes_to_track: FrozenSet[str] = frozenset(config.CLASSES_TO_TRACK)
    min_detection_confidence: Optional[float] = None
    max_cosine_distance: float = config.DEEPSORT_MAX_DIST
    max_iou_distance: float = config.DEEPSORT_MAX_IOU_DISTANCE
    max_age: int = config.DEEPSORT_MAX_AGE
    n_init: int = config.DEEPSORT_N_INIT
    include_regions: Tuple[Tuple[Tuple[int, int], ...], ...] = ()
    exclude_regions: Tuple[Tuple[Tuple[int, int], ...], ...] = ()

    def __post_init__(self):
        if isinstance(self.classes_to_track, str):
            raise ValueError("classes_to_track is a set of class names, not one string")
        classes = frozenset(self.classes_to_track)
        unknown = classes - set(config.CLASSES)
        if unknown:
            raise ValueError("unknown class names: %s" % sorted(unknown))
        object.__setattr__(self, "classes_to_track", classes)
        for name in ("conf_threshold", "nms_threshold", "min_detection_confidence"):
            v = getattr(self, name)
            if v is not None and not (isinstance(v, (int, float)) and 0.0 <= v <= 1.0):
                raise ValueError("%s must be a number in [0, 1], got %r" % (name, v))
        for name in ("max_cosine_distance", "max_iou_distance"):
            v = getattr(self, name)
            if not (isinstance(v, (int, float)) and math.isfinite(v) and v >= 0):
                raise ValueError("%s must be finite and non-negative, got %r" % (name, v))
        if not (isinstance(self.max_age, int) and 1 <= self.max_age <= 255):
            raise ValueError("max_age must be an integer in 1..255, got %r" % (self.max_age,))
        if not (isinstance(self.n_init, int) and self.n_init >= 1):
            raise ValueError("n_init must be an integer >= 1, got %r" % (self.n_init,))
        for name in ("include_regions", "exclude_regions"):
            object.__setattr__(self, name, _polygons(getattr(self, name), name))
        if len(self.include_regions) + len(self.exclude_regions) > _lib.REGION_MAX_POLYGONS:
            raise ValueError("at most %d include and exclude polygons per stream, got %d"
                             % (_lib.REGION_MAX_POLYGONS, len(self.include_regions) + len(self.exclude_regions)))

    @classmethod
    def from_dict(cls, d, base: Optional["StreamSettings"] = None):
        """Settings from a dict of field names (e.g. a JSON object), over ``base`` (default: the config defaults)."""
        names = {f.name for f in fields(cls)}
        unknown = set(d) - names
        if unknown:
            raise ValueError("unknown stream settings: %s" % sorted(unknown))
        kw = {f.name: getattr(base or cls(), f.name) for f in fields(cls)}
        kw.update(d)
        return cls(**kw)

    def resolve(self):
        """(aicam_stream_filter, aicam_stream_assoc) of these settings."""
        score, min_conf = resolve_thresholds(self.conf_threshold, self.min_detection_confidence)
        lo, hi = config.tracked_class_mask(self.classes_to_track)
        return (_lib.StreamFilter(score, self.nms_threshold, min_conf, 0, lo, hi),
                _lib.StreamAssoc(float(self.max_cosine_distance), float(self.max_iou_distance), self.max_age, self.n_init))

    def has_regions(self):
        return bool(self.include_regions or self.exclude_regions)

    def resolve_region(self):
        """The aicam_stream_region of these settings' include and exclude polygons."""
        r = _lib.StreamRegion()
        polygons = [(0, p) for p in self.include_regions] + [(1, p) for p in self.exclude_regions]
        r.n_polygons = len(polygons)
        for i, (kind, pts) in enumerate(polygons):
            r.kind[i], r.n_vertices[i] = kind, len(pts)
            for k, (x, y) in enumerate(pts):
                r.xy[i][k][:] = [x, y]
        return r


def _filter_key(f):
    return (f.score_thr, f.iou_thr, f.min_confidence, f.class_mask_lo, f.class_mask_hi)


def _as_settings_list(indices, settings):
    indices = [int(i) for i in indices]
    if isinstance(settings, StreamSettings):
        settings = [settings] * len(indices)
    settings = list(settings)
    if len(settings) != len(indices) or not all(isinstance(s, StreamSettings) for s in settings):
        raise ValueError("configure_streams: one StreamSettings per index")
    return indices, settings


def _point(p, what):
    if not (isinstance(p, (tuple, list)) and len(p) == 2):
        raise ValueError("%s must be an (x, y) pair, got %r" % (what, p))
    for v in p:
        if isinstance(v, bool) or not isinstance(v, int):
            raise ValueError("%s: coordinates must be integers, got %r" % (what, p))
        if abs(v) > _lib.COUNT_MAX_COORD:
            raise ValueError("%s: coordinates are limited to +-2^20, got %r" % (what, p))
    return (int(p[0]), int(p[1]))


def _polygons(v, what):
    """A tuple of polygons (tuples of 3 to 32 integer (x, y) vertices) from a sequence of them."""
    if isinstance(v, str) or not isinstance(v, (tuple, list)):
        raise ValueError("%s must be a list of polygons, got %r" % (what, v))
    out = []
    for poly in v:
        if isinstance(poly, str) or not isinstance(poly, (tuple, list)):
            raise ValueError("%s: a polygon is a list of (x, y) vertices, got %r" % (what, poly))
        pts = tuple(_point(p, what + " vertex") for p in poly)
        if not 3 <= len(pts) <= _lib.COUNT_MAX_VERTICES:
            raise ValueError("%s: a polygon needs 3 to %d vertices, got %d" % (what, _lib.COUNT_MAX_VERTICES, len(pts)))
        out.append(pts)
    return tuple(out)


def _classes(classes):
    if classes is None:
        return None
    if isinstance(classes, str):
        raise ValueError("classes is a set of class names, not one string")
    classes = frozenset(classes)
    unknown = classes - set(config.CLASSES)
    if unknown:
        raise ValueError("unknown class names: %s" % sorted(unknown))
    return classes


def _from_dict(cls, d):
    if not isinstance(d, dict):
        raise ValueError("%s: expected an object, got %r" % (cls.__name__, d))
    unknown = set(d) - {f.name for f in fields(cls)}
    if unknown:
        raise ValueError("unknown %s fields: %s" % (cls.__name__, sorted(unknown)))
    return cls(**d)


@dataclass(frozen=True)
class CountingLine:
    """A counting line from ``a`` to ``b`` (integer frame pixels).  A track whose bottom-centre anchor passes from the
    left-hand side of a->b to its right-hand side (on screen, y pointing down) goes "in", the other way "out".
    ``classes``: the class names counted (None: the pipeline's tracked classes)."""
    a: Tuple[int, int]
    b: Tuple[int, int]
    name: Optional[str] = None
    classes: Optional[FrozenSet[str]] = None

    def __post_init__(self):
        object.__setattr__(self, "a", _point(self.a, "line end a"))
        object.__setattr__(self, "b", _point(self.b, "line end b"))
        if self.a == self.b:
            raise ValueError("a counting line needs two distinct ends, got %r twice" % (self.a,))
        if self.name is not None and not isinstance(self.name, str):
            raise ValueError("name must be a string, got %r" % (self.name,))
        object.__setattr__(self, "classes", _classes(self.classes))

    @classmethod
    def from_dict(cls, d):
        return _from_dict(cls, d)


@dataclass(frozen=True)
class CountingZone:
    """A counting zone: a polygon of 3 to 32 integer vertices (even-odd rule; may be concave or self-intersecting).
    ``classes`` as for CountingLine.  ``loiter_frames``: a track that stays in the zone for that many of its stream's
    frames raises one loiter event per visit (0: none); setting it turns dwell on for the stream (StreamCounting)."""
    points: Tuple[Tuple[int, int], ...]
    name: Optional[str] = None
    classes: Optional[FrozenSet[str]] = None
    loiter_frames: Optional[int] = None

    def __post_init__(self):
        if isinstance(self.points, str) or not hasattr(self.points, "__len__"):
            raise ValueError("points must be a sequence of (x, y) pairs")
        pts = tuple(_point(p, "zone vertex") for p in self.points)
        if not 3 <= len(pts) <= _lib.COUNT_MAX_VERTICES:
            raise ValueError("a zone needs 3 to %d vertices, got %d" % (_lib.COUNT_MAX_VERTICES, len(pts)))
        object.__setattr__(self, "points", pts)
        if self.name is not None and not isinstance(self.name, str):
            raise ValueError("name must be a string, got %r" % (self.name,))
        object.__setattr__(self, "classes", _classes(self.classes))
        v = self.loiter_frames
        if v is not None and (isinstance(v, bool) or not isinstance(v, int) or not 0 <= v <= _lib.DWELL_MAX_LOITER):
            raise ValueError("loiter_frames must be an integer in 0..2^30, got %r" % (v,))

    @classmethod
    def from_dict(cls, d):
        return _from_dict(cls, d)


@dataclass(frozen=True)
class StreamCounting:
    """One stream's counting lines and zones (at most 16 of each).  Unnamed ones are called ``line{i}`` / ``zone{i}``
    after their index; names are unique within the stream.  ``dwell``: also measure how long tracks stay in the zones
    (include/aicam.h, "Dwell"); a zone with ``loiter_frames`` turns it on."""
    lines: Tuple[CountingLine, ...] = ()
    zones: Tuple[CountingZone, ...] = ()
    dwell: bool = False

    def __post_init__(self):
        lines, zones = tuple(self.lines), tuple(self.zones)
        if not all(isinstance(x, CountingLine) for x in lines) or not all(isinstance(x, CountingZone) for x in zones):
            raise ValueError("lines must be CountingLine and zones CountingZone objects")
        if not isinstance(self.dwell, bool):
            raise ValueError("dwell must be true or false, got %r" % (self.dwell,))
        if any(x.loiter_frames is not None for x in zones):
            object.__setattr__(self, "dwell", True)
        if len(lines) > _lib.COUNT_MAX_LINES or len(zones) > _lib.COUNT_MAX_ZONES:
            raise ValueError("at most %d lines and %d zones per stream" % (_lib.COUNT_MAX_LINES, _lib.COUNT_MAX_ZONES))
        lines = tuple(x if x.name is not None else replace(x, name="line%d" % i) for i, x in enumerate(lines))
        zones = tuple(x if x.name is not None else replace(x, name="zone%d" % i) for i, x in enumerate(zones))
        for kind, items in (("line", lines), ("zone", zones)):
            names = [x.name for x in items]
            if len(set(names)) != len(names):
                raise ValueError("%s names must be unique within a stream: %s" % (kind, names))
        object.__setattr__(self, "lines", lines)
        object.__setattr__(self, "zones", zones)

    @classmethod
    def from_dict(cls, d):
        """From ``{"lines": [{"a": [x, y], "b": [x, y], "name": .., "classes": [..]}], "zones": [{"points": [[x, y],
        ..], "loiter_frames": n, ..}], "dwell": true}`` (e.g. a JSON object)."""
        if not isinstance(d, dict):
            raise ValueError("StreamCounting: expected an object, got %r" % (d,))
        unknown = set(d) - {"lines", "zones", "dwell"}
        if unknown:
            raise ValueError("unknown counting fields: %s" % sorted(unknown))

        def items(key, kind):
            v = d.get(key, [])
            if not isinstance(v, list):
                raise ValueError("%s must be a list" % key)
            return tuple(kind.from_dict(x) for x in v)
        return cls(items("lines", CountingLine), items("zones", CountingZone), d.get("dwell", False))

    def resolve(self, default_classes):
        """The aicam_stream_counting of this geometry; lines and zones without classes count ``default_classes``."""
        g = _lib.StreamCounting()
        g.n_lines, g.n_zones = len(self.lines), len(self.zones)
        for i, x in enumerate(self.lines):
            g.line[i][:] = [x.a[0], x.a[1], x.b[0], x.b[1]]
            g.line_class_mask[i][:] = config.tracked_class_mask(x.classes if x.classes is not None else default_classes)
        for i, x in enumerate(self.zones):
            g.zone_n[i] = len(x.points)
            for k, (px, py) in enumerate(x.points):
                g.zone_xy[i][k][:] = [px, py]
            g.zone_class_mask[i][:] = config.tracked_class_mask(x.classes if x.classes is not None else default_classes)
        return g

    def resolve_dwell(self):
        """The aicam_stream_dwell of these settings."""
        d = _lib.StreamDwell()
        d.enabled = int(self.dwell)
        for i, x in enumerate(self.zones):
            d.loiter_frames[i] = x.loiter_frames or 0
        return d


class _DeviceArray:
    """A library-owned device array as torch sees it (__cuda_array_interface__); holds the handle's owner alive."""

    def __init__(self, owner, ptr, shape, typestr):
        self.owner = owner
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


class _CounterHandle:
    def __init__(self, lib, device, n_streams, max_tracks, max_events):
        self.lib, self.h = lib, C.c_void_p()
        _lib.check(lib.aicam_counter_create(device.index or 0, n_streams, max_tracks, max_events, C.byref(self.h)))

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.aicam_counter_destroy(self.h)
            self.h = None


class StreamCounter:
    """Owner of an ``aicam_counter``: line crossings and zone entries of ``n_streams`` streams, counted on the device
    from a tracker's reported rows.  The outputs are device tensors over the library's buffers (stable, so a captured
    step keeps writing them; they stay valid while any of them or the counter lives):
      line_counts int64 [S, 16, 2, 80] (in, out per class), zone_counts int64 [S, 16, 2, 80] (entries, exits),
      occupancy int32 [S, 16, 80], row_zones int32 [S, T] (zone bits of row n of out_tracks), events int32
      [S, max_events, 4] (kind 0 line in, 1 line out, 2 zone entry, 3 zone exit; index; track id; class) and
      event_count int32 [S] of the last step.
    Dwell (after the first ``set_dwell``; None before): visits, frames_total, frames_max int64 [S, 16, 80] (completed
    visits per zone and class, their summed and largest durations in frames), row_dwell int32 [S, T, 16] (frames since
    entry of row n's open visit in each zone, -1 for none), dwell_events int32 [S, max_events, 5] (kind 0 visit
    completed, 1 loiter; zone; track id; class; frames) and dwell_event_count int32 [S] of the last step."""

    def __init__(self, device, n_streams: int, max_tracks: int, max_events: int = 1024):
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.S, self.T, self.E = int(n_streams), int(max_tracks), int(max_events)
        self._handle = _CounterHandle(self.lib, self.device, self.S, self.T, self.E)
        o = _lib.CounterOutput()
        _lib.check(self.lib.aicam_counter_outputs(self._handle.h, C.byref(o)))
        L, Z, K = _lib.COUNT_MAX_LINES, _lib.COUNT_MAX_ZONES, _lib.COUNT_CLASSES

        def view(ptr, shape, typestr):
            return torch.as_tensor(_DeviceArray(self._handle, ptr, shape, typestr), device=self.device)
        self.line_counts = view(o.line_counts, (self.S, L, 2, K), "<i8")
        self.zone_counts = view(o.zone_counts, (self.S, Z, 2, K), "<i8")
        self.occupancy = view(o.occupancy, (self.S, Z, K), "<i4")
        self.row_zones = view(o.row_zones, (self.S, self.T), "<i4")  # (bits 0..15: never negative)
        self.events = view(o.events, (self.S, self.E, 4), "<i4")
        self.event_count = view(o.event_count, (self.S,), "<i4")
        self.visits = self.frames_total = self.frames_max = self.row_dwell = None
        self.dwell_events = self.dwell_event_count = None

    @property
    def handle(self):
        return self._handle.h

    @property
    def has_dwell(self):
        """Dwell is set up (some set_dwell call has succeeded): the dwell buffers exist."""
        return self.visits is not None

    def set_dwell(self, indices, settings: Sequence["_lib.StreamDwell"]):
        """Streams ``indices`` take the dwell ``settings`` (aicam_stream_dwell records); a stream that was disabled and
        is enabled starts its dwell state, an enabled one whose thresholds change keeps it."""
        n = len(indices)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aicam_counter_set_dwell(self.handle, (C.c_int32 * n)(*indices), (_lib.StreamDwell * n)(*settings),
                                                        n, _lib.stream_ptr(self.device)))
        if self.visits is None and n:
            o = _lib.CounterDwellOutput()
            _lib.check(self.lib.aicam_counter_dwell_outputs(self.handle, C.byref(o)))
            Z, K = _lib.COUNT_MAX_ZONES, _lib.COUNT_CLASSES

            def view(ptr, shape, typestr):
                return torch.as_tensor(_DeviceArray(self._handle, ptr, shape, typestr), device=self.device)
            self.visits = view(o.visits, (self.S, Z, K), "<i8")
            self.frames_total = view(o.frames_total, (self.S, Z, K), "<i8")
            self.frames_max = view(o.frames_max, (self.S, Z, K), "<i8")
            self.row_dwell = view(o.row_dwell, (self.S, self.T, Z), "<i4")
            self.dwell_events = view(o.events, (self.S, self.E, 5), "<i4")
            self.dwell_event_count = view(o.event_count, (self.S,), "<i4")

    def dwell_step(self, out_tracks, out_count, row_slot, present=None):
        """The dwell step of the rows ``step`` has just counted (same arguments, after it)."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aicam_counter_dwell_step(self.handle, _lib.ptr(out_tracks), _lib.ptr(out_count), row_slot,
                                                         present, _lib.stream_ptr(self.device)))

    def dwell_overflow(self):
        """Sticky per-stream flags: some dwell step had more events than max_events (the dwell counters stayed exact)."""
        import numpy as np
        f = np.zeros(self.S, np.int32)
        _lib.check(self.lib.aicam_counter_dwell_overflow(self.handle, _lib.ptr(f)))
        return f

    def set_streams(self, indices, geometry: Sequence["_lib.StreamCounting"]):
        """Streams ``indices`` take ``geometry`` (aicam_stream_counting records); their counts and tracks restart."""
        n = len(indices)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aicam_counter_set_streams(self.handle, (C.c_int32 * n)(*indices),
                                                          (_lib.StreamCounting * n)(*geometry), n,
                                                          _lib.stream_ptr(self.device)))

    def step(self, out_tracks, out_count, row_slot, present=None):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aicam_counter_step(self.handle, _lib.ptr(out_tracks), _lib.ptr(out_count), row_slot, present,
                                                   _lib.stream_ptr(self.device)))

    def reset_streams(self, mask):
        """Restart the streams whose entry of the device int32 [S] mask is non-zero."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aicam_counter_reset_streams(self.handle, _lib.ptr(mask), _lib.stream_ptr(self.device)))

    def overflow(self):
        """Sticky per-stream flags: some step had more events than max_events (the counters stayed exact)."""
        import numpy as np
        f = np.zeros(self.S, np.int32)
        _lib.check(self.lib.aicam_counter_overflow(self.handle, _lib.ptr(f)))
        return f


def frame_geometry(frames: torch.Tensor):
    """(n, h, w, is_nv12) of a batch of frames: [n, H, W, 3] packed BGR or [n, H*3/2, W] NV12."""
    if frames.dtype != torch.uint8 or not frames.is_contiguous():
        raise _lib.AicamError(-1, "frames must be a contiguous uint8 tensor")
    if frames.dim() == 4 and frames.shape[3] == 3:
        return frames.shape[0], frames.shape[1], frames.shape[2], False
    if frames.dim() == 3 and frames.shape[1] % 3 == 0:
        return frames.shape[0], frames.shape[1] * 2 // 3, frames.shape[2], True
    raise _lib.AicamError(-1, "frames must be [n, H, W, 3] (BGR) or [n, H*3/2, W] (NV12)")


def is_frame_list(frames) -> bool:
    return isinstance(frames, (list, tuple))


class FrameTable:
    """Owner of an ``aicam_frame_table``: per-stream frames of any size, row pitch and surface format for one batched
    step.  ``set(frames)`` takes a list of uint8 CUDA tensors, each ``[H, W, 3]`` BGR or ``[H*3/2, W]`` NV12, whose rows
    are contiguous (a view into a larger surface is fine: its row stride is the pitch).  The library may read every
    plane as rows * pitch bytes, so a view's last row must be followed by the rest of its pitch inside the same storage.
    A ``None`` entry marks that stream ABSENT for the step (a dropped or late frame, a source that has ended): it is not
    read, its detection row is empty and its tracker state does not change.  ``present`` is the device i32[capacity] 0/1
    mask of the last set (a stable pointer that captured steps read)."""

    def __init__(self, device, capacity: int, max_frame_hw=(2160, 3840)):
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.capacity, self.max_frame_hw = int(capacity), tuple(max_frame_hw)
        self._h = C.c_void_p()
        _lib.check(self.lib.aicam_frame_table_create(self.device.index or 0, self.capacity, self.max_frame_hw[0],
                                                     self.max_frame_hw[1], C.byref(self._h)))
        self._descs = (_lib.FrameDesc * self.capacity)()
        self._present = (C.c_uint8 * self.capacity)()
        self.n = 0
        self.n_present = 0
        self.frames = []
        self.present_ptr = C.c_void_p(self.lib.aicam_frame_table_present(self._h))
        self.filters = None
        self.region_test = False  # some entry has had polygons: each table crop step launches the region test

    def set_filters(self, filters: Optional[Sequence["_lib.StreamFilter"]]):
        """Per-entry detection and filter settings (aicam_frame_table_set_filters): entry i < len(filters) is detected
        and filtered with filters[i] from the next ``set`` on; None clears them (every entry uses the entry points'
        arguments again)."""
        n = len(filters) if filters else 0
        arr = (_lib.StreamFilter * n)(*filters) if n else None
        _lib.check(self.lib.aicam_frame_table_set_filters(self._h, arr, n))
        self.filters = list(filters) if n else None

    def set_regions(self, indices, regions: Sequence["_lib.StreamRegion"]):
        """Entries ``indices`` take ``regions`` (aicam_stream_region records; n_polygons 0 clears one) from the next
        step on, eager or captured; the other entries keep theirs.  One copy on the current stream."""
        indices = [int(i) for i in indices]
        n = len(indices)
        if len(regions) != n:
            raise ValueError("set_regions: one region per index")
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aicam_frame_table_set_regions(self._h, (C.c_int32 * n)(*indices),
                                                              (_lib.StreamRegion * n)(*regions), n,
                                                              _lib.stream_ptr(self.device)))
        self.region_test |= any(r.n_polygons > 0 for r in regions)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self.lib.aicam_frame_table_destroy(h)
            self._h = None

    @staticmethod
    def describe(frame: torch.Tensor):
        """(h, w, pitch, kind) of one frame; kind 0 BGR, 1 NV12."""
        if frame.dtype != torch.uint8 or not frame.is_cuda:
            raise _lib.AicamError(-1, "frames must be uint8 CUDA tensors")
        if frame.dim() == 3 and frame.shape[2] == 3 and frame.stride(2) == 1 and frame.stride(1) == 3:
            return frame.shape[0], frame.shape[1], frame.stride(0), 0
        if frame.dim() == 2 and frame.shape[0] % 3 == 0 and frame.stride(1) == 1:
            return frame.shape[0] * 2 // 3, frame.shape[1], frame.stride(0), 1
        raise _lib.AicamError(-1, "each frame must be [H, W, 3] (BGR) or [H*3/2, W] (NV12) with contiguous rows")

    def set(self, frames: Sequence[torch.Tensor]):
        n = len(frames)
        if n > self.capacity:
            raise _lib.AicamError(-4, "%d frames exceed the frame table's capacity %d" % (n, self.capacity))
        for i, f in enumerate(frames):
            d = self._descs[i]
            self._present[i] = f is not None
            if f is None:
                d.data, d.chroma, d.h, d.w, d.pitch, d.kind = None, None, 0, 0, 0, 0
                continue
            if f.device != self.device:
                raise _lib.AicamError(-1, "frame %d is not on %s" % (i, self.device))
            h, w, pitch, kind = self.describe(f)
            if f.storage_offset() + f.shape[0] * pitch > f.untyped_storage().nbytes():
                raise _lib.AicamError(-1, "frame %d: its %d rows of %d bytes (the pitch) run past the end of its storage"
                                      % (i, f.shape[0], pitch))
            d.data, d.h, d.w, d.pitch, d.kind = f.data_ptr(), h, w, pitch, kind
            d.chroma = f.data_ptr() + h * pitch if kind == 1 else None
        n_present = sum(f is not None for f in frames)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aicam_frame_table_set_present(self._h, self._descs,
                                                              self._present if n_present < n else None, n,
                                                              _lib.stream_ptr(self.device)))
        self.n, self.n_present = n, n_present
        self.frames = list(frames)  # kept alive while work that reads the table may be in flight

    @property
    def handle(self):
        return self._h


class BatchDetector:
    """K1-K4 + detect() post-processing for ``batch`` frames of one size."""

    def __init__(self, engine_path, batch: int, device=None, conf_threshold=config.YOLO_CONF_THRESHOLD,
                 nms_threshold=config.YOLO_NMS_THRESHOLD, topk=config.YOLO_TOPK,
                 max_candidates=config.YOLO_MAX_CANDIDATES, max_frame_hw=(2160, 3840)):
        self.max_frame_hw = tuple(max_frame_hw)
        self.frame_table = None  # created on the first list of frames
        self.engine = TRTEngine(engine_path, device, max_batch=batch, topk=topk,
                                score_threshold=resolve_thresholds(conf_threshold)[0],
                                nms_threshold=nms_threshold, max_candidates=max_candidates)
        if self.engine.kind != _lib.KIND_YOLOV8:
            raise RuntimeError("BatchDetector needs a yolov8 weight blob")
        self.lib = _lib.load()
        self.device = self.engine.device
        self.batch, self.topk = batch, topk
        self.conf_threshold = conf_threshold
        e, dev = self.engine, self.device
        self.num_dets = torch.zeros(batch, dtype=torch.int32, device=dev)
        self.boxes_lb = torch.zeros((batch, topk, 4), dtype=torch.float32, device=dev)
        self.boxes = torch.zeros((batch, topk, 4), dtype=torch.float32, device=dev)
        self.scores = torch.zeros((batch, topk), dtype=torch.float32, device=dev)
        self.labels = torch.zeros((batch, topk), dtype=torch.int32, device=dev)
        self._nms = _lib.NmsParams(e.score_threshold, e.nms_threshold, topk, e.max_candidates, 0, 0)
        # 0: NHWC4 input (aicam_preprocess format 1), 1: 2x2 pixel blocks (format 2), 2: 4x4 pixel blocks (format 3, yolov8n)
        self._s2d = int(self.lib.aicam_engine_accepts_s2d(e.handle))

    def detect(self, frames):
        """frames: uint8 cuda [n<=batch, H, W, 3] BGR, or [n, H*3/2, W] NV12 (Y plane + interleaved UV plane, the
        surface format of hardware decoders: half the bytes), or a list of n such frames ([H_s, W_s, 3] / [H_s*3/2, W_s])
        of any sizes and kinds, where None marks an absent frame (its row reports no detections; the network runs over
        the present frames only).  Returns device tensors (num_dets [n],
        boxes [n,topk,4] in frame pixels, scores [n,topk], labels [n,topk]); views of internal
        buffers, valid until the next call; asynchronous on the current stream."""
        if is_frame_list(frames):
            if self.frame_table is None:
                self.frame_table = FrameTable(self.device, self.batch, self.max_frame_hw)
            self.frame_table.set(frames)
            return self.detect_table(self.frame_table)
        n, h, w, nv12 = frame_geometry(frames)
        pre = self.lib.aicam_preprocess_nv12 if nv12 else self.lib.aicam_preprocess
        if n > self.batch:
            raise _lib.AicamError(-4, "detect: %d frames exceed the detector's batch %d" % (n, self.batch))
        e, st = self.engine, _lib.stream_ptr(self.device)
        with torch.cuda.device(self.device):
            # same bytes in 2x2 / 4x4 pixel blocks (formats 2 / 3): the stride-2 stem runs as a stride-1 window over the blocks
            _lib.check(pre(_lib.ptr(frames), n, h, w, 1 + self._s2d, _lib.ptr(e._nhwc), st))
            self._nms.frame_h, self._nms.frame_w = h, w
            # network + decode (fused into the Detect-head epilogues) + NMS + un-letterboxing: one entry
            _lib.check(self.lib.aicam_yolo_detect(
                e.handle, _lib.ptr(e._nhwc), self._s2d, n, C.byref(self._nms),
                _lib.ptr(e._head) if e._head is not None else None, _lib.ptr(self.num_dets),
                _lib.ptr(self.boxes_lb), _lib.ptr(self.boxes), _lib.ptr(self.scores), _lib.ptr(self.labels),
                _lib.ptr(e._ws), e._ws.numel(), st))
        return self.num_dets[:n], self.boxes[:n], self.scores[:n], self.labels[:n]

    def detect_table(self, table: FrameTable):
        """detect() on the frames a FrameTable holds (each un-letterboxed with its own size); capturable."""
        n = table.n
        if n > self.batch:
            raise _lib.AicamError(-4, "detect: %d frames exceed the detector's batch %d" % (n, self.batch))
        e, st = self.engine, _lib.stream_ptr(self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aicam_preprocess_table(table.handle, 1 + self._s2d, _lib.ptr(e._nhwc), st))
            _lib.check(self.lib.aicam_yolo_detect_table(
                e.handle, _lib.ptr(e._nhwc), self._s2d, table.handle, C.byref(self._nms),
                _lib.ptr(e._head) if e._head is not None else None, _lib.ptr(self.num_dets),
                _lib.ptr(self.boxes_lb), _lib.ptr(self.boxes), _lib.ptr(self.scores), _lib.ptr(self.labels),
                _lib.ptr(e._ws), e._ws.numel(), st))
        return self.num_dets[:n], self.boxes[:n], self.scores[:n], self.labels[:n]

    def launches_per_step(self, frame_list=False):
        # K1 + network + NMS (+ the decode kernel when the engine cannot decode inside its Detect-head epilogues); over a frame
        # table K1 is two launches (row-staged and per-pixel), both made whatever the frame sizes
        k1 = 2 if frame_list else 1
        return k1 + self.engine.launches_per_forward() + (1 if self.engine.fused_decode else 2)


class BatchTracker:
    """K5-K12 for ``n_streams`` independent streams (one DeepSORT state each)."""

    def __init__(self, reid_engine_path, n_streams: int, device=None, max_dets=config.YOLO_TOPK,
                 max_tracks: int = 256, max_crops: Optional[int] = None,
                 max_cosine_distance=config.DEEPSORT_MAX_DIST, nn_budget=config.DEEPSORT_NN_BUDGET,
                 max_iou_distance=config.DEEPSORT_MAX_IOU_DISTANCE, max_age=config.DEEPSORT_MAX_AGE,
                 n_init=config.DEEPSORT_N_INIT, min_detection_confidence=config.DEEPSORT_MIN_CONFIDENCE,
                 max_frame_hw=(2160, 3840), classes_to_track=config.CLASSES_TO_TRACK):
        self.max_frame_hw = tuple(max_frame_hw)
        self.frame_table = None  # created on the first list of frames
        self.max_crops = int(max_crops if max_crops is not None else min(n_streams * max_dets, 4096))
        self.reid = TRTEngine(reid_engine_path, device, max_batch=self.max_crops)
        if self.reid.kind != _lib.KIND_REID:
            raise RuntimeError("BatchTracker needs a reid weight blob")
        if nn_budget is None:
            raise RuntimeError("nn_budget=None (unbounded galleries) is not supported on the device")
        self.lib = _lib.load()
        self.device = dev = self.reid.device
        self.S, self.K, self.T = n_streams, max_dets, max_tracks
        self.min_conf = float(min_detection_confidence)
        self.classes_to_track = frozenset(classes_to_track)
        self.assoc_defaults = dict(max_cosine_distance=float(max_cosine_distance), max_iou_distance=float(max_iou_distance),
                                   max_age=int(max_age), n_init=int(n_init))
        self.F = self.reid.feature_dim
        cfg = _lib.TrackerConfig(n_streams, max_tracks, max_dets, self.F, float(max_cosine_distance),
                                 float(max_iou_distance), int(max_age), int(n_init), int(nn_budget), dev.index)
        self._h = C.c_void_p()
        _lib.check(self.lib.aicam_tracker_create(C.byref(cfg), C.byref(self._h)))
        S, K = n_streams, max_dets
        i32 = dict(dtype=torch.int32, device=dev)
        self.det_index = torch.zeros((S, K), **i32)
        self.det_count = torch.zeros(S, **i32)
        self.crop_slot = torch.zeros((S, K), **i32)
        self.crop_rect = torch.zeros((self.max_crops, 5), **i32)
        self.crop_count = torch.zeros(2, **i32)  # [crops written, high-water mark of crops wanted]
        # crops go straight into the layout the engine's first kernel reads (NHWC8 for the fused stem)
        self._nhwc8 = bool(self.lib.aicam_engine_accepts_nhwc8(self.reid.handle))
        self.crops = torch.zeros((self.max_crops, config.REID_INPUT_SHAPE[0], config.REID_INPUT_SHAPE[1],
                                  8 if self._nhwc8 else 4),
                                 dtype=torch.bfloat16, device=dev)
        self.feats = torch.zeros((self.max_crops, self.F), dtype=torch.float32, device=dev)
        self.out_tracks = torch.zeros((S, max_tracks, 6), **i32)
        self.out_conf = torch.zeros((S, max_tracks), dtype=torch.float32, device=dev)
        self.out_count = torch.zeros(S, **i32)
        self.row_slots = C.c_void_p(self.lib.aicam_tracker_row_slots(self._h))  # device i32 [S, T]: slot of each row
        self._reset_mask = torch.zeros(S, **i32)
        self._mask = config.tracked_class_mask(self.classes_to_track)
        # per-stream confidence and class mask of configure_streams (None: every stream uses the constructor's); a list
        # step hands them to the frame table, a stacked step whose streams differ goes through the table
        self._filters = None
        self._routed = False
        # per-stream regions of configure_streams (None until some stream has had polygons), handed to the frame table
        self._regions = None
        # optional running totals (crops, reported tracks) kept on the device, for benchmarks: no host sync
        self.count_stats = False
        self.crop_total = torch.zeros(1, dtype=torch.int64, device=dev)
        self.track_total = torch.zeros(1, dtype=torch.int64, device=dev)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self.lib.aicam_tracker_destroy(h)
            self._h = None

    def reset(self):
        _lib.check(self.lib.aicam_tracker_reset(self._h, _lib.stream_ptr(self.device)))
        self.crop_count.zero_()

    def reset_streams(self, indices):
        """Reset the given streams to a fresh tracker's state (no tracks, ids from 1), e.g. when a slot is handed to
        another camera or clip; every other stream keeps its tracks.  One kernel launch on the current stream."""
        mask = torch.zeros(self.S, dtype=torch.int32)
        for i in indices:
            if not 0 <= int(i) < self.S:
                raise _lib.AicamError(-1, "reset_streams: stream %d out of range" % int(i))
            mask[int(i)] = 1
        with torch.cuda.device(self.device):
            self._reset_mask.copy_(mask)
            _lib.check(self.lib.aicam_tracker_reset_streams(self._h, _lib.ptr(self._reset_mask), _lib.stream_ptr(self.device)))

    def configure_streams(self, indices, settings):
        """Give the streams ``indices`` their own association settings (max_cosine_distance, max_iou_distance, max_age,
        n_init) and crop filter (minimum confidence, tracked classes), from the next step on.  The other streams, and
        the tracks of these, are untouched; a track keeps the n_init and max_age it was created with, as in the
        reference.  ``settings``: one StreamSettings per index, or one for all."""
        indices, settings = _as_settings_list(indices, settings)
        resolved = [s.resolve() for s in settings]
        assoc = (_lib.StreamAssoc * len(indices))(*[a for _, a in resolved])
        idx = (C.c_int32 * len(indices))(*indices)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aicam_tracker_set_stream_assoc(self._h, idx, assoc, len(indices), _lib.stream_ptr(self.device)))
        base = _lib.StreamFilter(0.0, 0.0, self.min_conf, 0, self._mask[0], self._mask[1])
        filters = self._filters or [base] * self.S
        for i, (f, _) in zip(indices, resolved):
            filters[i] = f
        self._filters = filters
        if self._regions is not None or any(s.has_regions() for s in settings):
            if self._regions is None:
                self._regions = [_lib.StreamRegion() for _ in range(self.S)]
            for i, s in zip(indices, settings):
                self._regions[i] = s.resolve_region()
            if self.frame_table is not None:
                self.frame_table.set_regions(indices, [self._regions[i] for i in indices])
        key = _filter_key(base)[2:]
        # (once some stream has had a region, every step runs the region test over the table)
        self._routed = any(_filter_key(f)[2:] != key for f in filters) or self._regions is not None

    def update(self, frames, num_dets, boxes, scores, labels):
        """One frame per stream.  frames uint8 cuda [S,H,W,3] BGR or [S,H*3/2,W] NV12, or a list of S frames of any
        sizes and kinds, None for a stream that has no frame this step (see BatchDetector.detect: its state is left as it
        is and its out_count is 0); detections as BatchDetector
        returns them ([S], [S,K,4], [S,K], [S,K]).  Returns device (out_tracks [S,T,6] int32 =
        x1,y1,x2,y2,id,class, out_conf [S,T], out_count [S]); asynchronous."""
        if not is_frame_list(frames) and self._routed:
            frame_geometry(frames)
            frames = list(frames.unbind(0))  # streams filter differently: one table entry per stream
        if is_frame_list(frames):
            if self.frame_table is None:
                self.frame_table = FrameTable(self.device, self.S, self.max_frame_hw)
                if self._regions is not None:
                    self.frame_table.set_regions(range(self.S), self._regions)
            if self._filters is not None:
                self.frame_table.set_filters(self._filters)
            self.frame_table.set(frames)
            return self.update_table(self.frame_table, num_dets, boxes, scores, labels)
        S, h, w, nv12 = frame_geometry(frames)
        crops_fn = self.lib.aicam_reid_crops_nv12 if nv12 else self.lib.aicam_reid_crops
        if S != self.S or boxes.shape[1] != self.K:
            raise _lib.AicamError(-4, "update: expected %d streams x %d detections" % (self.S, self.K))
        st = _lib.stream_ptr(self.device)
        with torch.cuda.device(self.device):
            _lib.check(crops_fn(
                _lib.ptr(frames), S, h, w, _lib.ptr(boxes), _lib.ptr(scores), _lib.ptr(labels), _lib.ptr(num_dets),
                self.K, self.min_conf, self._mask[0], self._mask[1], 2 if self._nhwc8 else 1, self.max_crops,
                _lib.ptr(self.det_index),
                _lib.ptr(self.det_count), _lib.ptr(self.crop_slot), _lib.ptr(self.crop_rect), _lib.ptr(self.crops),
                _lib.ptr(self.crop_count), st))
        return self._reid_and_step(boxes, scores, labels, None)

    def update_table(self, table: FrameTable, num_dets, boxes, scores, labels):
        """update() on the frames a FrameTable holds (one per stream, absent ones included); capturable, and a captured
        step follows the presence of each later ``table.set``."""
        if table.n != self.S or boxes.shape[1] != self.K:
            raise _lib.AicamError(-4, "update: expected %d streams x %d detections" % (self.S, self.K))
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aicam_reid_crops_table(
                table.handle, _lib.ptr(boxes), _lib.ptr(scores), _lib.ptr(labels), _lib.ptr(num_dets),
                self.K, self.min_conf, self._mask[0], self._mask[1], 2 if self._nhwc8 else 1, self.max_crops,
                _lib.ptr(self.det_index), _lib.ptr(self.det_count), _lib.ptr(self.crop_slot), _lib.ptr(self.crop_rect),
                _lib.ptr(self.crops), _lib.ptr(self.crop_count), _lib.stream_ptr(self.device)))
        return self._reid_and_step(boxes, scores, labels, table.present_ptr)

    def _reid_and_step(self, boxes, scores, labels, present):
        st = _lib.stream_ptr(self.device)
        with torch.cuda.device(self.device):
            fwd = self.lib.aicam_reid_forward_nhwc8 if self._nhwc8 else self.lib.aicam_reid_forward
            _lib.check(fwd(self.reid.handle, _lib.ptr(self.crops), self.max_crops, _lib.ptr(self.crop_count),
                           _lib.ptr(self.feats), st))
            # present: the frame table's device mask (absent streams keep their state), or None on the tensor path
            _lib.check(self.lib.aicam_tracker_step_present(
                self._h, _lib.ptr(boxes), _lib.ptr(scores), _lib.ptr(labels), self.K, _lib.ptr(self.det_index),
                _lib.ptr(self.det_count), _lib.ptr(self.crop_slot), _lib.ptr(self.feats), present,
                _lib.ptr(self.out_tracks), _lib.ptr(self.out_conf), _lib.ptr(self.out_count), st))
            if self.count_stats:
                self.crop_total += self.crop_count[0:1]
                self.track_total += self.out_count.sum()
        return self.out_tracks, self.out_conf, self.out_count

    def overflow(self):
        import numpy as np
        f = np.zeros(self.S, np.int32)
        _lib.check(self.lib.aicam_tracker_overflow(self._h, _lib.ptr(f)))
        # bit 2 (every stream): some step wanted more ReID crops than max_crops, so detections lost their feature
        if int(self.crop_count[1].item()) > self.max_crops:
            f |= 4
        return f

    def snapshot(self, stream_index=0):
        import numpy as np
        ints = np.zeros((self.T, 7), np.int32)
        floats = np.zeros((self.T, 25), np.float32)
        n = self.lib.aicam_tracker_snapshot(self._h, stream_index, _lib.ptr(ints), _lib.ptr(floats), self.T)
        if n < 0:
            _lib.check(n)
        return ints[:n], floats[:n]

    def launches_per_step(self):
        # (no NHWC8 repack kernel; the region test once some stream has had a region)
        return (2 + self.reid.launches_per_forward() - (1 if self._nhwc8 else 0) + 3 +
                (1 if self._regions is not None else 0))


class TrackingPipeline:
    """detect + track for ``n_streams`` streams; one call per time step.  A step takes one stacked tensor of frames of
    one size, or a list with one frame per stream of any sizes (up to ``max_frame_hw``), pitches and kinds (BGR / NV12),
    where None marks a stream without a frame at this step: its tracks are neither predicted nor aged, and it reports
    no tracks.  (Aging tracks through a dropped frame is a different policy, not this one.)"""

    def __init__(self, yolo_engine_path, reid_engine_path, n_streams: int, device=None, max_tracks: int = 256,
                 max_crops: Optional[int] = None, conf_threshold=config.YOLO_CONF_THRESHOLD, topk=config.YOLO_TOPK,
                 max_candidates=config.YOLO_MAX_CANDIDATES, max_frame_hw=(2160, 3840),
                 nms_threshold=config.YOLO_NMS_THRESHOLD, stream_settings: Optional[Sequence[StreamSettings]] = None,
                 counting: Optional[Sequence[Optional[StreamCounting]]] = None, max_events: int = 1024, **tracker_kw):
        self.detector = BatchDetector(yolo_engine_path, n_streams, device, conf_threshold=conf_threshold,
                                      nms_threshold=nms_threshold, topk=topk, max_candidates=max_candidates,
                                      max_frame_hw=max_frame_hw)
        # detect() drops detections below conf_threshold before update() sees them (yolo_detector.py:131); on the
        # device that filter and DeepSORT's own (deepsort_tracker.py:88-95) are one comparison
        tracker_kw["min_detection_confidence"] = resolve_thresholds(conf_threshold,
                                                                    tracker_kw.get("min_detection_confidence"))[1]
        self.tracker = BatchTracker(reid_engine_path, n_streams, self.detector.device, max_dets=self.detector.topk,
                                    max_tracks=max_tracks, max_crops=max_crops, **tracker_kw)
        self.device = self.detector.device
        self.n_streams = n_streams
        # the frames of a list step: set once, read by the detector and the tracker
        self.frame_table = FrameTable(self.device, n_streams, max_frame_hw)
        # the settings the constructor's arguments amount to, and each stream's current ones
        self.default_settings = StreamSettings(conf_threshold, nms_threshold, self.tracker.classes_to_track,
                                               self.tracker.min_conf, **self.tracker.assoc_defaults)
        self.settings = [self.default_settings] * n_streams
        self._routed = False  # some stream detects or filters differently: stacked steps go through the frame table
        if stream_settings is not None:
            self.configure_streams(range(n_streams), stream_settings)
        # line and zone counting: the counter exists (and each step launches it) once some stream has counting
        self.counter: Optional[StreamCounter] = None
        self.counting = [None] * n_streams
        self.max_events = int(max_events)
        if counting is not None:
            self.configure_counting(range(n_streams), counting)

    def configure_streams(self, indices, settings):
        """Give the streams ``indices`` their own StreamSettings (one per index, or one for all) from the next step on,
        with or without a reset, whether the step runs eager or from a captured graph (call it between replays, like
        ``frame_table.set``).  The other streams are untouched; a stream's existing tracks keep the n_init and max_age
        they were created with, as in the reference.  The first settings with regions add the region test to every step
        from then on; a step captured before that does not include it, so capture again after the first region."""
        indices, settings = _as_settings_list(indices, settings)
        for i in indices:
            if not 0 <= i < self.n_streams:
                raise _lib.AicamError(-1, "configure_streams: stream %d out of range" % i)
        self.tracker.configure_streams(indices, settings)
        for i, st in zip(indices, settings):
            self.settings[i] = st
        filters = [st.resolve()[0] for st in self.settings]
        self.frame_table.set_filters(filters)
        if self.frame_table.region_test or any(st.has_regions() for st in settings):
            self.frame_table.set_regions(indices, [st.resolve_region() for st in settings])
        base = _filter_key(self.default_settings.resolve()[0])
        self._routed = any(_filter_key(f) != base for f in filters) or self.frame_table.region_test

    def configure_counting(self, indices, counting):
        """Give the streams ``indices`` their counting lines and zones (one StreamCounting or None per index, or one for
        all; None: no counting) from the next step on, eager or from a captured graph (call it between replays, like
        ``frame_table.set``).  Their counters and occupancy restart at zero and their tracks are counted from their next
        report on, as first reports; the other streams are untouched.  The first call that gives a stream counting
        creates the counter: from then on every step launches it once after the tracker.  A step captured before that
        does not include the counter, so capture again after turning counting on.  Dwell (StreamCounting.dwell, or a zone
        with loiter_frames) is set or cleared with the geometry; the first stream with dwell adds the dwell launch to
        every step from then on, and likewise a step captured before it does not include it."""
        indices = [int(i) for i in indices]
        if counting is None or isinstance(counting, StreamCounting):
            counting = [counting] * len(indices)
        counting = list(counting)
        if len(counting) != len(indices) or not all(c is None or isinstance(c, StreamCounting) for c in counting):
            raise ValueError("configure_counting: one StreamCounting (or None) per index")
        for i in indices:
            if not 0 <= i < self.n_streams:
                raise _lib.AicamError(-1, "configure_counting: stream %d out of range" % i)
        if self.counter is None:
            if all(c is None for c in counting):
                return
            self.counter = StreamCounter(self.device, self.n_streams, self.tracker.T, self.max_events)
        geometry = [(c or StreamCounting()).resolve(self.tracker.classes_to_track) for c in counting]
        self.counter.set_streams(indices, geometry)
        if self.counter.has_dwell or any(c is not None and c.dwell for c in counting):
            self.counter.set_dwell(indices, [(c or StreamCounting()).resolve_dwell() for c in counting])
        for i, c in zip(indices, counting):
            self.counting[i] = c

    def step(self, frames: Union[torch.Tensor, Sequence[torch.Tensor]]) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        if not is_frame_list(frames) and self._routed:
            frame_geometry(frames)
            frames = list(frames.unbind(0))  # streams detect or filter differently: one table entry per stream
        if is_frame_list(frames):
            self.frame_table.set(frames)
            return self.step_table()
        num, boxes, scores, labels = self.detector.detect(frames)
        return self._count(self.tracker.update(frames, num, boxes, scores, labels), None)

    def step_table(self) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """One step over the frames ``frame_table`` holds.  Launches depend only on the stream count and the size
        bound, so a captured step_table() stays valid when ``frame_table.set`` changes the frames, or which of them are
        present, between replays."""
        num, boxes, scores, labels = self.detector.detect_table(self.frame_table)
        return self._count(self.tracker.update_table(self.frame_table, num, boxes, scores, labels),
                           self.frame_table.present_ptr)

    def _count(self, tables, present):
        if self.counter is not None:
            out_tracks, _, out_count = tables
            self.counter.step(out_tracks, out_count, self.tracker.row_slots, present)
            if self.counter.has_dwell:
                self.counter.dwell_step(out_tracks, out_count, self.tracker.row_slots, present)
        return tables

    def counts(self):
        """Per stream, the cumulative counts since the stream's counting was last set or reset, and the occupancy of
        its last step: ``{"lines": {name: {"in": {class: n}, "out": {...}}}, "zones": {name: {"entered": {...},
        "exited": {...}, "occupancy": {...}}}}``, zeros omitted ({} for a stream without counting).  Synchronises."""
        out = [{} for _ in range(self.n_streams)]
        if self.counter is None:
            return out
        lc, zc, occ = (x.cpu().numpy() for x in (self.counter.line_counts, self.counter.zone_counts, self.counter.occupancy))

        def by_class(v):
            return {config.CLASSES[k]: int(v[k]) for k in range(len(v)) if v[k]}
        for s, c in enumerate(self.counting):
            if c is None:
                continue
            out[s] = {"lines": {x.name: {"in": by_class(lc[s, i, 0]), "out": by_class(lc[s, i, 1])} for i, x in enumerate(c.lines)},
                      "zones": {x.name: {"entered": by_class(zc[s, i, 0]), "exited": by_class(zc[s, i, 1]),
                                         "occupancy": by_class(occ[s, i])} for i, x in enumerate(c.zones)}}
        return out

    def dwell(self):
        """Per stream with dwell, the visits completed since the stream's dwell state last started (its counting was set
        or reset, or dwell turned on), per zone and class: ``{zone name: {"visits": {class: n}, "frames_total": {...},
        "frames_max": {...}}}``, durations in the stream's own frames, zeros omitted ({} for a stream without dwell).
        Synchronises."""
        out = [{} for _ in range(self.n_streams)]
        if self.counter is None or not self.counter.has_dwell:
            return out
        v, ft, fm = (x.cpu().numpy() for x in (self.counter.visits, self.counter.frames_total, self.counter.frames_max))

        def by_class(a):
            return {config.CLASSES[k]: int(a[k]) for k in range(len(a)) if a[k]}
        for s, c in enumerate(self.counting):
            if c is not None and c.dwell:
                out[s] = {x.name: {"visits": by_class(v[s, i]), "frames_total": by_class(ft[s, i]),
                                   "frames_max": by_class(fm[s, i])} for i, x in enumerate(c.zones)}
        return out

    def reset_streams(self, indices, settings=None):
        """Hand the given stream slots to new sources: their trackers restart (no tracks, ids from 1) and so do their
        counts and dwell, the other streams and the captured step are untouched.  The slots keep their settings and counting
        geometry, or take ``settings`` (as configure_streams)."""
        if settings is not None:
            self.configure_streams(indices, settings)
        self.tracker.reset_streams(indices)
        if self.counter is not None:  # (ids restart at 1: a new track must not continue an old one's counting state)
            self.counter.reset_streams(self.tracker._reset_mask)

    def launches_per_step(self, frame_list=False):
        """Kernel launches of one step: of a stacked tensor, or of a list of frames (frame_list=True), absent frames
        or not.  A stacked tensor runs as a list while streams detect or filter differently or once some stream has had a
        region; the region test adds one from then on, the counter one, dwell one more."""
        return (self.detector.launches_per_step(frame_list or self._routed) + self.tracker.launches_per_step() +
                (1 if self.counter is not None else 0) + (1 if self.counter is not None and self.counter.has_dwell else 0))
