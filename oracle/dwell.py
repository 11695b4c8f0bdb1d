"""Dwell oracle: how long tracks stay in counting zones, and loiter alerts, per stream, restated in plain Python integers.

The rules are those of include/aicam.h ("Dwell"), which csrc/counting.cu implements on the device:
  clock   each stream with dwell enabled has a frame clock f, the number of its present steps since its dwell state last
          started, this step included; the state starts when dwell is enabled and again when the stream's counting is
          set or reset (``reset``).  An absent step does not advance it and changes nothing.
  state   per track: a bit set of zones with an open visit, a bit set of visits already alerted, the clock at each open
          visit's entry.  A track's first report starts from no open visit.
  per row and zone z, with in = bit z of the row's zone bits (oracle.counting's membership, its row_zones):
          class not in the zone's mask: the visit state of z is left as it is and the row reports -1 for z;
          in, no open visit: a visit opens with entry = f;
          not in, open visit: it closes with duration d = f - entry: visits += 1, frames_total += d, frames_max raised to
            d, and a visit event;
          in, open visit, L = loiter_frames[z] > 0, f - entry >= L, not yet alerted: a loiter event, the visit alerted.
  A track not reported at a step keeps its open visits, and their clock keeps running.
Like oracle/counting.py this keeps its per-track state by (stream, track id) where the device keeps it by (stream,
tracker slot): a live track keeps its slot and a deleted id never returns, so the device's first report of a new id in a
reused slot, which drops the previous occupant's visits, is here a new id without state.

``Dwell(counter)`` reads the geometry and the row_zones of an ``oracle.counting.Counter``: call ``counter.step(rows,
present)`` and then ``dwell.step(rows, present)`` with the same arguments, and ``dwell.reset(s)`` with every
``counter.set_stream(s, ..)`` or ``counter.reset(s)``.
"""
import numpy as np

from .counting import MAX_ZONES, NCLS, class_in

VISIT, LOITER = 0, 1


class Dwell:
    """Dwell state, counters (``visits``, ``frames_total``, ``frames_max``), the events of the last step (kept to
    ``max_events``), ``row_dwell`` of the last step and the sticky overflow flags, mirroring the device outputs."""

    def __init__(self, counter, max_events):
        self.counter = counter
        self.S, self.E = counter.S, max_events
        self.enabled = [False] * self.S
        self.loiter = [[0] * MAX_ZONES for _ in range(self.S)]
        self.visits = np.zeros((self.S, MAX_ZONES, NCLS), np.int64)
        self.frames_total = np.zeros((self.S, MAX_ZONES, NCLS), np.int64)
        self.frames_max = np.zeros((self.S, MAX_ZONES, NCLS), np.int64)
        self.overflow = np.zeros(self.S, np.int32)
        self.clock = [0] * self.S
        self.events = [[] for _ in range(self.S)]
        self.row_dwell = [[] for _ in range(self.S)]
        self.tracks = [{} for _ in range(self.S)]  # id -> [open bits, alerted bits, {zone: entry}]

    def set_dwell(self, s, enabled, loiter_frames=()):
        """Enable or disable stream s with per-zone loiter thresholds; enabling a disabled stream starts its state."""
        if enabled and not self.enabled[s]:
            self.reset(s)
        self.enabled[s] = bool(enabled)
        self.loiter[s] = list(loiter_frames) + [0] * (MAX_ZONES - len(loiter_frames))

    def reset(self, s):
        """Restart stream s's dwell state (settings kept)."""
        self.visits[s] = 0
        self.frames_total[s] = 0
        self.frames_max[s] = 0
        self.overflow[s] = 0
        self.clock[s] = 0
        self.events[s] = []
        self.row_dwell[s] = []
        self.tracks[s] = {}

    def step(self, rows, present=None):
        for s in range(self.S):
            if (present is not None and not present[s]) or not self.enabled[s]:
                self.events[s] = []
                continue
            self._stream(s, rows[s])

    def _stream(self, s, rows):
        self.clock[s] += 1
        f = self.clock[s]
        zones = self.counter.geometry[s][1]
        row_zones = self.counter.row_zones[s]
        events, row_dwell = [], []
        for r, row in enumerate(rows):
            tid, cls = int(row[4]), int(row[5])
            st = self.tracks[s].setdefault(tid, [0, 0, {}])
            dwell = [-1] * MAX_ZONES
            for z, (_, mask) in enumerate(zones):
                if not class_in(mask, cls):
                    continue
                bit = 1 << z
                if (row_zones[r] >> z) & 1:
                    if not st[0] & bit:
                        st[0] |= bit
                        st[1] &= ~bit
                        st[2][z] = f
                    dwell[z] = f - st[2][z]
                    L = self.loiter[s][z]
                    if L > 0 and dwell[z] >= L and not st[1] & bit:
                        st[1] |= bit
                        events.append((LOITER, z, tid, cls, dwell[z]))
                elif st[0] & bit:
                    d = f - st[2][z]
                    st[0] &= ~bit
                    st[1] &= ~bit
                    self.visits[s, z, cls] += 1
                    self.frames_total[s, z, cls] += d
                    self.frames_max[s, z, cls] = max(self.frames_max[s, z, cls], d)
                    events.append((VISIT, z, tid, cls, d))
            row_dwell.append(dwell)
        if len(events) > self.E:
            self.overflow[s] = 1
        self.events[s] = events[:self.E]
        self.row_dwell[s] = row_dwell
