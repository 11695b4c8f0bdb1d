"""Counting oracle: line crossings and zone entries per stream, restated in plain Python integers.

The rules are those of include/aicam.h ("Counting"), which csrc/counting.cu implements on the device.  This restatement
keeps its per-track state by (stream, track id) where the device keeps it by (stream, tracker slot): a live track keeps
its slot and a deleted id never returns, so the two are the same state, and every comparison against the device also
checks that.  Geometry per stream: ``lines`` = [((ax, ay), (bx, by), (mask_lo, mask_hi))], ``zones`` = [(points,
(mask_lo, mask_hi))], integer frame pixels.
"""
import numpy as np

MAX_LINES, MAX_ZONES, NCLS = 16, 16, 80
ANCHOR_LIMIT = 1 << 24
LINE_IN, LINE_OUT, ZONE_ENTRY, ZONE_EXIT = 0, 1, 2, 3


def _clamp(v):
    return max(-ANCHOR_LIMIT, min(ANCHOR_LIMIT, v))


def anchor(x1, y1, x2, y2):
    """Bottom centre of a row, doubled: (x1 + x2, 2 * y2), each clamped to [-2^24, 2^24]."""
    return _clamp(int(x1) + int(x2)), _clamp(2 * int(y2))


def side(a, b, p):
    """+1 when the doubled point p is strictly on the positive side of the doubled line a->b, else -1."""
    return 1 if (b[0] - a[0]) * (p[1] - a[1]) - (b[1] - a[1]) * (p[0] - a[0]) > 0 else -1


def crossing(a, b, p0, p1):
    """LINE_IN, LINE_OUT or None for a move p0 -> p1 (all doubled)."""
    s0, s1 = side(a, b, p0), side(a, b, p1)
    if s0 == s1:
        return None
    dx, dy = p1[0] - p0[0], p1[1] - p0[1]
    da = dx * (a[1] - p0[1]) - dy * (a[0] - p0[0])
    db = dx * (b[1] - p0[1]) - dy * (b[0] - p0[0])
    if (da > 0 and db > 0) or (da < 0 and db < 0):
        return None
    return LINE_IN if s1 > 0 else LINE_OUT


def inside(points, p):
    """Even-odd rule with half-open edges; points and p doubled."""
    px, py = p
    result = False
    n = len(points)
    for i in range(n):
        xi, yi = points[i]
        xj, yj = points[i - 1]
        if (yi > py) != (yj > py):
            # px < xi + (py - yi) * (xj - xi) / (yj - yi), without the division
            lhs, rhs, d = (px - xi) * (yj - yi), (py - yi) * (xj - xi), yj - yi
            if (lhs < rhs) if d > 0 else (lhs > rhs):
                result = not result
    return result


def class_in(mask, cls):
    lo, hi = mask
    return 0 <= cls < NCLS and ((lo >> cls) & 1 if cls < 64 else (hi >> (cls - 64)) & 1) == 1


class Counter:
    """``n_streams`` streams; ``step(rows, present)`` takes each stream's reported rows (x1, y1, x2, y2, id, class) of one
    step.  Counters, occupancy, ``row_zones``, the events of the last step (kept to ``max_events``) and the sticky
    overflow flags mirror the device outputs."""

    def __init__(self, n_streams, max_events):
        self.S, self.E = n_streams, max_events
        self.geometry = [([], []) for _ in range(n_streams)]
        self.line_counts = np.zeros((n_streams, MAX_LINES, 2, NCLS), np.int64)
        self.zone_counts = np.zeros((n_streams, MAX_ZONES, 2, NCLS), np.int64)
        self.occupancy = np.zeros((n_streams, MAX_ZONES, NCLS), np.int64)
        self.overflow = np.zeros(n_streams, np.int32)
        self.events = [[] for _ in range(n_streams)]
        self.row_zones = [[] for _ in range(n_streams)]
        self.tracks = [{} for _ in range(n_streams)]  # id -> (doubled anchor, zone bits)

    def set_stream(self, s, lines, zones):
        self.geometry[s] = (list(lines), list(zones))
        self.reset(s)

    def reset(self, s):
        self.line_counts[s] = 0
        self.zone_counts[s] = 0
        self.occupancy[s] = 0
        self.overflow[s] = 0
        self.events[s] = []
        self.row_zones[s] = []
        self.tracks[s] = {}

    def step(self, rows, present=None):
        for s in range(self.S):
            if present is not None and not present[s]:
                self.events[s] = []
                continue
            self._stream(s, rows[s])

    def _stream(self, s, rows):
        lines, zones = self.geometry[s]
        lines2 = [((2 * a[0], 2 * a[1]), (2 * b[0], 2 * b[1]), m) for a, b, m in lines]
        zones2 = [([(2 * x, 2 * y) for x, y in pts], m) for pts, m in zones]
        events, row_zones = [], []
        self.occupancy[s] = 0
        for x1, y1, x2, y2, tid, cls in rows:
            tid, cls = int(tid), int(cls)
            p = anchor(x1, y1, x2, y2)
            prev = self.tracks[s].get(tid)
            if prev is not None:
                for li, (a, b, m) in enumerate(lines2):
                    kind = crossing(a, b, prev[0], p)
                    if kind is not None and class_in(m, cls):
                        self.line_counts[s, li, kind, cls] += 1
                        events.append((kind, li, tid, cls))
            was = prev[1] if prev is not None else 0
            now = 0
            for zi, (pts, m) in enumerate(zones2):
                isin = inside(pts, p)
                now |= int(isin) << zi
                if not class_in(m, cls):
                    continue
                if isin:
                    self.occupancy[s, zi, cls] += 1
                if isin != bool((was >> zi) & 1):
                    self.zone_counts[s, zi, 0 if isin else 1, cls] += 1
                    events.append((ZONE_ENTRY if isin else ZONE_EXIT, zi, tid, cls))
            self.tracks[s][tid] = (p, now)
            row_zones.append(now)
        if len(events) > self.E:
            self.overflow[s] = 1
        self.events[s] = events[:self.E]
        self.row_zones[s] = row_zones
