"""Dwell on the device (dwell_kernel in csrc/counting.cu through aicam_counter_set_dwell / _dwell_step, StreamCounter, the
pipeline's configure_counting and --counting), each compared bit for bit with oracle/dwell.py on oracle/counting.py's
zone membership.  The oracle keeps its state by track id where the device keeps it by tracker slot."""
import ctypes as C
import json
import multiprocessing
import os
from dataclasses import replace

import numpy as np
import pytest
import torch

import test_gpu_counting as TC
from oracle import counting as O
from oracle import dwell as D

DEV = torch.device("cuda:0")
gpu = pytest.mark.gpu
NZ = 16
COUNTING_OUTPUTS = ("line_counts", "zone_counts", "occupancy", "event_count", "events", "row_zones")
DWELL_OUTPUTS = ("visits", "frames_total", "frames_max", "dwell_event_count", "dwell_events", "row_dwell")


def _L():
    from ai_camera_b200 import _lib as L
    return L


def _dwell(enabled, loiter=()):
    d = _L().StreamDwell()
    d.enabled = int(enabled)
    for z, v in enumerate(loiter):
        d.loiter_frames[z] = v
    return d


def assert_dwell_same(dev, oracle, rows, present, what):
    """Dwell counters, the last step's events and (for enabled present streams) row_dwell equal the oracle's."""
    torch.cuda.synchronize()
    assert np.array_equal(dev.visits.cpu().numpy(), oracle.visits), what
    assert np.array_equal(dev.frames_total.cpu().numpy(), oracle.frames_total), what
    assert np.array_equal(dev.frames_max.cpu().numpy(), oracle.frames_max), what
    ec, ev, rd = dev.dwell_event_count.cpu().numpy(), dev.dwell_events.cpu().numpy(), dev.row_dwell.cpu().numpy()
    for s in range(len(rows)):
        want = oracle.events[s]
        assert ec[s] == len(want), (what, s)
        assert [tuple(e) for e in ev[s, :ec[s]].tolist()] == want, (what, s)
        if oracle.enabled[s] and (present is None or present[s]):
            assert rd[s, :len(rows[s])].tolist() == oracle.row_dwell[s], (what, s)


class Pair:
    """Two device counters fed the same host rows, one with dwell and one without, next to the oracle."""

    def __init__(self, S, T, E):
        from ai_camera_b200.pipeline import StreamCounter
        self.S, self.T, self.E = S, T, E
        self.dev = StreamCounter(DEV, S, T, E)
        self.plain = StreamCounter(DEV, S, T, E)
        self.counting = O.Counter(S, E)
        self.oracle = D.Dwell(self.counting, E)
        i32 = dict(dtype=torch.int32, device=DEV)
        self.out_tracks = torch.zeros((S, T, 6), **i32)
        self.out_count = torch.zeros(S, **i32)
        self.row_slot = torch.zeros((S, T), **i32)
        self.present = torch.ones(S, **i32)
        self.mask = torch.zeros(S, **i32)

    def set_streams(self, indices, geoms):
        for c in (self.dev, self.plain):
            c.set_streams(indices, [TC._record(*g) for g in geoms])
        for i, g in zip(indices, geoms):
            self.counting.set_stream(i, *g)
            self.oracle.reset(i)

    def set_dwell(self, indices, enabled, loiters):
        self.dev.set_dwell(indices, [_dwell(e, l) for e, l in zip(enabled, loiters)])
        for i, e, l in zip(indices, enabled, loiters):
            self.oracle.set_dwell(i, e, l)

    def reset_streams(self, indices):
        m = np.zeros(self.S, np.int32)
        m[list(indices)] = 1
        self.mask.copy_(torch.from_numpy(m))
        for c in (self.dev, self.plain):
            c.reset_streams(self.mask)
        for i in indices:
            self.counting.reset(i)
            self.oracle.reset(i)

    def step(self, rows, slots, present=None, oracle=True):
        ot = np.zeros((self.S, self.T, 6), np.int32)
        rs = np.full((self.S, self.T), -1, np.int32)
        oc = np.zeros(self.S, np.int32)
        for s in range(self.S):
            oc[s] = len(rows[s])
            if oc[s]:
                ot[s, :oc[s]] = rows[s]
                rs[s, :oc[s]] = slots[s]
        self.out_tracks.copy_(torch.from_numpy(ot))
        self.out_count.copy_(torch.from_numpy(oc))
        self.row_slot.copy_(torch.from_numpy(rs))
        if present is not None:
            self.present.copy_(torch.from_numpy(np.asarray(present, np.int32)))
        args = (self.out_tracks, self.out_count, C.c_void_p(self.row_slot.data_ptr()),
                None if present is None else C.c_void_p(self.present.data_ptr()))
        self.dev.step(*args)
        self.dev.dwell_step(*args)
        self.plain.step(*args)
        if oracle:
            self.counting.step(rows, present)
            self.oracle.step(rows, present)

    def assert_counting_unaffected(self, what):
        torch.cuda.synchronize()
        for name in COUNTING_OUTPUTS:
            assert torch.equal(getattr(self.dev, name), getattr(self.plain, name)), (what, name)


class DwellFleet:
    """Synthetic tracker output for long runs: per stream, live tracks in slots that linger, are reported or missed,
    change class now and then, die and are born into free slots with new ids; anchors on a coarse grid (ties with the
    zones' vertices), now and then far outside the frame."""

    def __init__(self, rng, S, T, grid, extent):
        self.rng, self.S, self.T, self.grid, self.extent = rng, S, T, grid, extent
        self.live = [{} for _ in range(S)]  # slot -> [id, x, y, cls]
        self.next_id = [1] * S

    def step(self, fill=0.8):
        rng, g = self.rng, self.grid
        rows, slots = [], []
        for s in range(self.S):
            live = self.live[s]
            for slot in list(live):
                if rng.random() < 0.02:
                    del live[slot]
            free = [k for k in range(self.T) if k not in live]
            rng.shuffle(free)
            for slot in free[:max(0, int(self.T * fill) - len(live))]:
                live[slot] = [self.next_id[s], int(rng.integers(0, self.extent // g)) * g,
                              int(rng.integers(0, self.extent // g)) * g, int(rng.choice([0, 1, 2, 3, 5, 7, 79]))]
                self.next_id[s] += 1
            rep = [k for k in live if rng.random() < 0.75]
            rng.shuffle(rep)
            r = []
            for k in rep:
                t = live[k]
                if rng.random() < 0.5:
                    t[1] += int(rng.integers(-1, 2)) * g
                    t[2] += int(rng.integers(-1, 2)) * g
                if rng.random() < 0.03:
                    t[3] = int(rng.choice([0, 2, 79]))
                x, y = t[1], t[2]
                if rng.random() < 0.005:
                    x, y = int(rng.choice([-1, 1])) * (1 << 30), int(rng.choice([-1, 1])) * (1 << 29)
                half = int(rng.integers(0, 30))
                r.append((x - half, y - 40, x + half + int(rng.integers(0, 2)), y, t[0], t[3]))
            rows.append(r)
            slots.append(rep)
        return rows, slots


# ---- the fuzz at the maxima ---------------------------------------------------------------------------------------------

def _fuzz_case(seed=11, S=64, T=256, steps=300):
    """Rows, slots, presence and a schedule of set, enable, threshold and reset calls for every step."""
    rng = np.random.default_rng(seed)
    grid, extent = 16, 640
    geoms = [TC._random_geometry(rng, grid, extent) for _ in range(S)]
    choices = [0, 1, 2, 3, 4, 6, 10, 20, 50]
    loiters = [[int(v) for v in rng.choice(choices, NZ)] for _ in range(S)]
    fleet = DwellFleet(rng, S, T, grid, extent)
    data = []
    for t in range(steps):
        rows, slots = fleet.step()
        present = (rng.random(S) < 0.85).astype(np.int32).tolist() if t % 4 else None
        data.append((rows, slots, present))
    # step -> list of (call, stream, argument)
    sched = {0: [("dwell", s, (s != S - 1, loiters[s])) for s in range(S)]}
    sched.setdefault(steps // 3, []).append(("dwell", S - 1, (True, loiters[S - 1])))        # enabled mid-stream
    sched.setdefault(steps // 3 + 20, []).append(("dwell", 30, (False, loiters[30])))       # disabled ...
    sched.setdefault(steps // 2 + 30, []).append(("dwell", 30, (True, loiters[30])))        # ... and enabled again
    for s in range(8):                                                                       # thresholds change
        sched.setdefault(steps // 2, []).append(("dwell", s, (True, [int(v) for v in rng.choice(choices, NZ)])))
    sched.setdefault(2 * steps // 3, []).append(("reset", 10, None))
    sched.setdefault(2 * steps // 3, []).append(("reset", 11, None))
    sched.setdefault(2 * steps // 3 + 10, []).append(("set", 20, TC._random_geometry(rng, grid, extent)))
    return geoms, data, sched


def _oracle_stream(args):
    """One stream of the fuzz through the oracle (in a worker process): per step (events, row_dwell as an array or None,
    overflow flag), and the counters every 25 steps.  args: (geometry, [(rows, present or None)] per step, {step: [(call,
    argument)]}, max_events)."""
    geom, data, sched, E = args
    c = O.Counter(1, E)
    c.set_stream(0, *geom)
    d = D.Dwell(c, E)
    out, counters = [], {}
    for t, (rows, present) in enumerate(data):
        for call, arg in sched.get(t, ()):
            if call == "dwell":
                d.set_dwell(0, *arg)
            elif call == "reset":
                c.reset(0)
                d.reset(0)
            else:
                c.set_stream(0, *arg)
                d.reset(0)
        p = None if present is None else [present]
        c.step([rows], p)
        d.step([rows], p)
        shown = d.enabled[0] and (p is None or p[0])
        out.append((list(d.events[0]), np.array(d.row_dwell[0], np.int32).reshape(-1, NZ) if shown else None,
                    bool(d.overflow[0])))
        if t % 25 == 24 or t == len(data) - 1:
            counters[t] = (d.visits[0].copy(), d.frames_total[0].copy(), d.frames_max[0].copy())
    return out, counters


@gpu
def test_fuzz_at_the_maxima_equals_the_oracle_and_leaves_counting_alone():
    S, T, steps = 64, 256, 300
    E = T * NZ  # (room for every event: the flags stay clear)
    geoms, data, sched = _fuzz_case(S=S, T=T, steps=steps)
    work = [(geoms[s], [(rows[s], None if present is None else present[s]) for rows, _, present in data],
             {t: [(call, arg) for call, i, arg in calls if i == s] for t, calls in sched.items()}, E) for s in range(S)]
    # (spawned workers: this process has threads, which a fork would copy in whatever state they are)
    with multiprocessing.get_context("spawn").Pool(max(1, min(S, os.cpu_count() or 1))) as pool:
        want = pool.map(_oracle_stream, work)
    p = Pair(S, T, E)
    p.set_streams(list(range(S)), geoms)
    kinds = np.zeros(2, np.int64)
    alerted_at = set()
    for t, (rows, slots, present) in enumerate(data):
        for call, i, arg in sched.get(t, ()):
            if call == "dwell":
                p.dev.set_dwell([i], [_dwell(*arg)])
            elif call == "reset":
                p.reset_streams([i])
            else:
                for c in (p.dev, p.plain):
                    c.set_streams([i], [TC._record(*arg)])
        p.step(rows, slots, present, oracle=False)
        torch.cuda.synchronize()
        ec, ev, rd = p.dev.dwell_event_count.cpu().numpy(), p.dev.dwell_events.cpu().numpy(), p.dev.row_dwell.cpu().numpy()
        for s in range(S):
            events, row_dwell, _ = want[s][0][t]
            assert ec[s] == len(events), (t, s)
            assert [tuple(e) for e in ev[s, :ec[s]].tolist()] == events, (t, s)
            if row_dwell is not None:
                assert np.array_equal(rd[s, :len(rows[s])], row_dwell), (t, s)
            for e in events:
                kinds[e[0]] += 1
                if e[0] == D.LOITER:
                    alerted_at.add(e[4])
        if t in want[0][1]:
            for name, k in (("visits", 0), ("frames_total", 1), ("frames_max", 2)):
                got = getattr(p.dev, name).cpu().numpy()
                for s in range(S):
                    assert np.array_equal(got[s], want[s][1][t][k]), (t, s, name)
        if t % 10 == 0 or t == steps - 1:
            p.assert_counting_unaffected("step %d" % t)
    assert (kinds > 1000).all(), kinds
    assert {1, 2} <= alerted_at and max(alerted_at) >= 50, sorted(alerted_at)  # (thresholds 1 and 2, and long visits)
    assert int(p.dev.frames_max.max()) > 50
    assert not p.dev.dwell_overflow().any() and not p.dev.overflow().any()
    assert not any(w[0][-1][2] for w in want)


# ---- overflow, rejected calls -------------------------------------------------------------------------------------------

ALL = ((1 << 64) - 1, (1 << 16) - 1)
SQ = [(0, 0), (100, 0), (100, 100), (0, 100)]


def _row(x, y, tid):
    return (x - 2, y - 10, x + 2, y, tid, 0)


@gpu
def test_event_overflow_truncates_in_order_and_keeps_counters():
    S, T, E = 3, 32, 5
    p = Pair(S, T, E)
    p.set_streams(list(range(S)), [([], [(SQ, ALL)])] * S)
    p.set_dwell(list(range(S)), [True] * S, [[1]] * S)
    # stream s has 4 * s tracks; they enter four at a time, stay one step (a loiter event each) and leave: at most four
    # counting events a step, up to eight dwell events
    n = [1, 4, 8]
    inside = lambda k, t: 2 * (k // 4) <= t < 2 * (k // 4) + 3  # noqa: E731
    for t in range(6):
        rows = [[_row(50 if inside(k, t) else 300, 50, k + 1) for k in range(n[s])] for s in range(S)]
        slots = [list(range(len(r))) for r in rows]
        p.step(rows, slots)
        assert_dwell_same(p.dev, p.oracle, rows, None, "step %d" % t)
        TC.assert_same(p.dev, p.counting, rows, None, "step %d" % t)
        p.assert_counting_unaffected("step %d" % t)
    assert p.oracle.overflow.tolist() == [0, 0, 1]
    assert p.dev.dwell_overflow().tolist() == [0, 0, 1]
    assert p.dev.overflow().tolist() == [0, 0, 0]  # counting's flag is its own
    assert int(p.dev.visits[2].sum()) == 8 and int(p.dev.frames_total[2].sum()) == 8 * 3
    p.reset_streams([2])
    assert p.dev.dwell_overflow().tolist() == [0, 0, 0] and int(p.dev.visits[2].sum()) == 0
    assert int(p.dev.visits[1].sum()) == 4


@gpu
def test_rejected_calls_change_nothing():
    S, T, E = 2, 16, 64
    rng = np.random.default_rng(5)
    lib = _L().load()
    L = _L()
    # a counter without dwell: a rejected call allocates nothing, and the dwell entry points refuse
    from ai_camera_b200.pipeline import StreamCounter
    c0 = StreamCounter(DEV, S, T, E)
    bad = _dwell(True, [-1])
    assert lib.aicam_counter_set_dwell(c0.handle, (C.c_int32 * 1)(0), (L.StreamDwell * 1)(bad), 1, None) == -1
    o = L.CounterDwellOutput()
    assert lib.aicam_counter_dwell_outputs(c0.handle, C.byref(o)) == -1
    assert lib.aicam_counter_dwell_step(c0.handle, C.c_void_p(1), C.c_void_p(1), C.c_void_p(1), None, None) == -1
    assert lib.aicam_counter_set_dwell(c0.handle, None, None, 0, None) == 0
    assert lib.aicam_counter_dwell_outputs(c0.handle, C.byref(o)) == -1
    assert not c0.has_dwell and c0.dwell_overflow().tolist() == [0, 0]

    a, b = Pair(S, T, E), Pair(S, T, E)
    geo = TC._random_geometry(rng, 8, 200, n_lines=2, n_zones=4, n_vert=5)
    for p in (a, b):
        p.set_streams([0, 1], [geo, geo])
        p.set_dwell([0, 1], [True, True], [[1, 2, 0, 3], [0, 0, 5, 1]])
    fleet = TC.Fleet(rng, S, T, 8, 200)
    steps = [fleet.step(0.5) for _ in range(10)]
    for p in (a, b):
        for rows, slots in steps[:5]:
            p.step(rows, slots)
    good = _dwell(False, [7])
    cases = [([0], [_dwell(2, [])]), ([0], [_dwell(True, [-1])]), ([1], [_dwell(True, [0] * 15 + [(1 << 30) + 1])]),
             ([2], [good]), ([-1], [good]), ([1, 0], [good, _dwell(True, [5, -3])])]
    torch.cuda.synchronize()
    before = lib.aicam_launch_count()
    for idx, recs in cases:
        n = len(idx)
        assert lib.aicam_counter_set_dwell(b.dev.handle, (C.c_int32 * n)(*idx), (L.StreamDwell * n)(*recs), n, None) == -1, idx
    assert lib.aicam_counter_set_dwell(b.dev.handle, None, None, 1, None) == -1
    assert lib.aicam_counter_set_dwell(b.dev.handle, (C.c_int32 * 1)(0), (L.StreamDwell * 1)(good), -1, None) == -1
    assert lib.aicam_counter_dwell_step(b.dev.handle, None, None, None, None, None) == -1
    assert lib.aicam_launch_count() == before
    for rows, slots in steps[5:]:
        for p in (a, b):
            p.step(rows, slots)
        torch.cuda.synchronize()
        for name in DWELL_OUTPUTS + COUNTING_OUTPUTS:
            assert torch.equal(getattr(a.dev, name), getattr(b.dev, name)), name
    assert_dwell_same(b.dev, b.oracle, steps[-1][0], None, "after the rejected calls")
    assert int(b.dev.visits.sum()) > 0


# ---- pipeline -----------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def blobs(tmp_path_factory):
    from ai_camera_b200 import synth
    return synth.make_blobs(str(tmp_path_factory.mktemp("blobs")))


@pytest.fixture(scope="module")
def bias(blobs):
    from ai_camera_b200 import synth
    return synth.shifted_class_bias(blobs[0], -0.6)


def _pipeline(blobs, bias, n, **kw):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import TrackingPipeline
    p = TrackingPipeline(blobs[0], blobs[1], n, max_tracks=128, n_init=1, **kw)
    synth.apply_class_bias(p.detector.engine, bias)
    return p


def _with_dwell(sc, loiter=None, dwell=True):
    """``sc`` with dwell, and the zones' loiter thresholds ``loiter`` (None: none)."""
    zones = sc.zones if loiter is None else tuple(replace(z, loiter_frames=l) for z, l in zip(sc.zones, loiter))
    return replace(sc, zones=zones, dwell=dwell or loiter is not None)


class PipeOracle:
    def __init__(self, pipe):
        self.pipe = pipe
        self.counting = O.Counter(pipe.n_streams, pipe.max_events)
        self.dwell = D.Dwell(self.counting, pipe.max_events)
        for s, c in enumerate(pipe.counting):
            self.configure(s, c)

    def configure(self, s, sc):
        """As configure_counting of stream s."""
        from ai_camera_b200.pipeline import StreamCounting
        sc = sc or StreamCounting()
        self.counting.set_stream(s, *TC._oracle_geometry(sc, self.pipe.tracker.classes_to_track))
        self.dwell.reset(s)
        self.dwell.set_dwell(s, sc.dwell, [z.loiter_frames or 0 for z in sc.zones])

    def step(self, rows, present):
        self.counting.step(rows, present)
        self.dwell.step(rows, present)


def _oracle_for(pipe):
    return PipeOracle(pipe)


@gpu
def test_pipeline_dwell_equals_the_oracle(blobs, bias):
    """Five streams: two with loiter thresholds, one with dwell and no threshold, one counting without dwell, one without
    counting; one stream absent at some steps.  Dwell equals the oracle over the pipeline's own rows, counting and the
    tracks are those of a pipeline without dwell, which launches one kernel less."""
    sizes = [(540, 960), (720, 1280), (540, 960), (480, 640), (540, 960)]
    S, T = len(sizes), 14
    videos = [TC._video(h, w, 500 + i, T) for i, (h, w) in enumerate(sizes)]
    base = [TC._counting(960, 540, 11), TC._counting(1280, 720, 12), TC._counting(960, 540, 13), None,
            TC._counting(960, 540, 14)]
    counting = [_with_dwell(base[0], [1, 3]), _with_dwell(base[1], [2, 0]), base[2], None, _with_dwell(base[4])]
    pipe = _pipeline(blobs, bias, S, counting=counting)
    plain = _pipeline(blobs, bias, S, counting=base)
    assert pipe.counter.has_dwell and not plain.counter.has_dwell
    oracle = _oracle_for(pipe)
    lib = _L().load()
    launches = {}
    kinds = np.zeros(2, np.int64)
    for t in range(T):
        frames = [None if (s == 1 and t in (4, 5, 9)) else videos[s][t] for s in range(S)]
        got = {}
        for name, p in (("pipe", pipe), ("plain", plain)):
            before = lib.aicam_launch_count()
            got[name] = [x.cpu().numpy() for x in p.step(frames)]
            launches.setdefault(name, set()).add(lib.aicam_launch_count() - before)
        for a, b in zip(got["pipe"], got["plain"]):
            assert np.array_equal(a, b), t
        for name in COUNTING_OUTPUTS:
            assert torch.equal(getattr(pipe.counter, name), getattr(plain.counter, name)), (t, name)
        present = [f is not None for f in frames]
        rows = TC._host_rows(got["pipe"][0], got["pipe"][2], S)
        oracle.step(rows, present)
        assert_dwell_same(pipe.counter, oracle.dwell, rows, present, "step %d" % t)
        for s in range(S):
            for e in oracle.dwell.events[s]:
                kinds[e[0]] += 1
    assert kinds[D.LOITER] > 0, kinds  # (completed visits are pinned in numbers by the fuzz)
    assert len(launches["plain"]) == 1 and launches["pipe"] == {n + 1 for n in launches["plain"]}
    assert pipe.launches_per_step() == plain.launches_per_step() + 1
    totals = pipe.dwell()
    assert totals[2] == totals[3] == {}
    from ai_camera_b200 import config
    for s in (0, 1, 4):
        for i, z in enumerate(counting[s].zones):
            for key in ("visits", "frames_total", "frames_max"):
                arr = getattr(oracle.dwell, key)[s, i]
                assert totals[s][z.name][key] == {config.CLASSES[k]: int(v) for k, v in enumerate(arr) if v}, (s, key)
    assert not pipe.counter.dwell_overflow().any()
    # a stacked step: the same dwell as the list step
    stacked = _pipeline(blobs, bias, 2, counting=[counting[0]] * 2)
    listed = _pipeline(blobs, bias, 2, counting=[counting[0]] * 2)
    for t in range(6):
        frames = [videos[0][t], videos[2][t]]
        stacked.step(torch.stack(frames))
        listed.step(frames)
        torch.cuda.synchronize()
        for name in DWELL_OUTPUTS:
            assert torch.equal(getattr(stacked.counter, name), getattr(listed.counter, name)), (t, name)


@gpu
def test_captured_step_follows_presence_counting_and_threshold_changes(blobs, bias):
    sizes = [(540, 960), (1080, 1920), (480, 640)]
    S, T = 3, 12
    videos = [TC._video(h, w, 530 + i, T) for i, (h, w) in enumerate(sizes)]
    masks = [[1, 1, 1], [1, 0, 1], [1, 1, 1], [0, 1, 1], [1, 1, 0], [1, 1, 1], [1, 1, 1], [0, 0, 1], [1, 1, 1],
             [1, 1, 1], [1, 0, 1], [1, 1, 1]]
    c0, c1, c2 = TC._counting(960, 540, 21), TC._counting(1920, 1080, 22), TC._counting(640, 480, 23)
    start = [_with_dwell(c0, [1, 2]), c1, _with_dwell(c2)]
    changes = {2: ([1], [_with_dwell(c1, [2, 1])]),                 # dwell on for a stream (its counting restarts)
               4: ([0], [_with_dwell(c0, [4, 0])]),                 # thresholds change (counting restarts too)
               6: ([2], [c2]),                                      # dwell off
               8: ([0, 2], [None, _with_dwell(c2, [1, 1])])}        # counting off; dwell on again
    g_pipe = _pipeline(blobs, bias, S, max_frame_hw=(1080, 1920), counting=start)
    e_pipe = _pipeline(blobs, bias, S, max_frame_hw=(1080, 1920), counting=start)
    g_pipe.step([v[0] for v in videos])
    torch.cuda.synchronize()
    g_pipe.reset_streams(range(S))
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        g_pipe.step_table()
    oracle = _oracle_for(e_pipe)
    events = 0
    for t in range(T):
        if t in changes:
            for p in (g_pipe, e_pipe):
                p.configure_counting(*changes[t])
            for s, sc in zip(*changes[t]):
                oracle.configure(s, sc)
        frames = [videos[s][t] if masks[t][s] else None for s in range(S)]
        g_pipe.frame_table.set(frames)
        g.replay()
        ot, _, on = [x.cpu().numpy() for x in e_pipe.step(frames)]
        torch.cuda.synchronize()
        for name in DWELL_OUTPUTS + COUNTING_OUTPUTS:
            assert torch.equal(getattr(g_pipe.counter, name), getattr(e_pipe.counter, name)), (t, name)
        rows = TC._host_rows(ot, on, S)
        oracle.step(rows, [bool(m) for m in masks[t]])
        assert_dwell_same(e_pipe.counter, oracle.dwell, rows, masks[t], "step %d" % t)
        events += int(e_pipe.counter.dwell_event_count.sum())
    assert events > 0
    assert g_pipe.dwell() == e_pipe.dwell()


@gpu
def test_resets_restart_dwell_of_the_selected_streams(blobs, bias):
    from ai_camera_b200.aicamera_tracker import run_batched
    S, T, R = 3, 10, 5
    videos = [TC._video(540, 960, 560 + i, T) for i in range(S)]
    sc = _with_dwell(TC._counting(960, 540, 27), [2, 1])
    pipe = _pipeline(blobs, bias, S, counting=[sc] * S)
    oracle = _oracle_for(pipe)
    for t in range(T):
        if t == R:
            before = pipe.counter.visits.clone()
            pipe.reset_streams([1])
            oracle.counting.reset(1)
            oracle.dwell.reset(1)
            torch.cuda.synchronize()
            assert int(pipe.counter.visits[1].sum()) == 0 and torch.equal(pipe.counter.visits[0], before[0])
        ot, _, on = [x.cpu().numpy() for x in pipe.step([v[t] for v in videos])]
        rows = TC._host_rows(ot, on, S)
        oracle.step(rows, None)
        assert_dwell_same(pipe.counter, oracle.dwell, rows, None, "step %d" % t)
    assert int(pipe.counter.visits.sum()) > 0
    # the refill loop: a slot handed to the next source restarts its dwell; the other slot keeps its own
    srcs = [[v.cpu().numpy() for v in videos[0]], [v.cpu().numpy() for v in videos[1][:4]]]
    refill = [[v.cpu().numpy() for v in videos[2][:5]]]
    pipe = _pipeline(blobs, bias, 2, counting=[sc] * 2)
    oracle = _oracle_for(pipe)

    def on_refill(slot, k):
        oracle.counting.reset(slot)
        oracle.dwell.reset(slot)

    def on_step(step, batch, table):
        ot, _, on = [x.numpy() for x in table]
        rows = TC._host_rows(ot, on, 2)
        present = [f is not None for f in batch]
        oracle.step(rows, present)
        assert_dwell_same(pipe.counter, oracle.dwell, rows, present, "refill step %d" % step)
    run_batched(srcs, pipe, on_step, until="all", refill=iter(refill), on_refill=on_refill)


@gpu
def test_cli_dwell_events_and_totals_equal_the_oracle_over_its_tracks(blobs, tmp_path):
    import cv2
    from ai_camera_b200 import config, synth, weights
    from ai_camera_b200.aicamera_tracker import load_counting, main, video_frames
    kind, params, tensors = weights.read_blob(blobs[0])
    tensors = dict(tensors)
    for n, b in synth.shifted_class_bias(blobs[0], synth.CLIP_LOGIT_SHIFT).items():
        tensors[n + ".bias"] = b
    yolo = weights.write_blob(str(tmp_path / "yolo_clip.aicw"), kind, params, tensors)
    clip = list(video_frames(TC.CLIP, 14))
    h, w = clip[0].shape[:2]
    paths = [TC._write_clip(tmp_path / "a.mp4", clip),
             TC._write_clip(tmp_path / "b.mp4", [cv2.resize(f, (640, 360)) for f in clip[:8]]),
             TC._write_clip(tmp_path / "c.mp4", clip[3:12])]
    def frame(w, h):  # (a box clipped to the frame's bottom edge has its anchor on y = h: keep it inside)
        return [[-8, -8], [w + 8, -8], [w + 8, h + 8], [-8, h + 8]]
    spec = {"default": {"zones": [{"points": [[0, 0], [w // 2, 0], [w // 2, h], [0, h]], "name": "left", "loiter_frames": 2},
                                  {"points": frame(w, h), "name": "all", "loiter_frames": 1}]},
            "b.mp4": {"zones": [{"points": frame(640, 360), "name": "frame"}], "dwell": True},
            "c.mp4": {"zones": [{"points": frame(w, h), "name": "all"}]}}
    (tmp_path / "c.json").write_text(json.dumps(spec))
    out = tmp_path / "out"
    for run_all in (False, True):
        argv = sum((["--input", p] for p in paths), []) + ["--streams", "2", "--counting", str(tmp_path / "c.json"),
                                                         "--output_dir", str(out), "--output_filename", "run%d" % run_all,
                                                         "--yolo_engine", yolo, "--reid_engine", blobs[1]]
        assert main(argv + (["--run_all_inputs"] if run_all else [])) == 0
        lines = [json.loads(l) for l in open(out / ("run%d.tracks.jsonl" % run_all))]
        counts = json.load(open(out / ("run%d.counts.json" % run_all)))
        get = load_counting(str(tmp_path / "c.json"))
        runs = [(os.path.basename(p), s) for s, p in enumerate(paths[:2])] if not run_all else \
            [(os.path.basename(p), None) for p in paths]
        assert [e["input"] for e in counts] == [n for n, _ in runs]
        total = 0
        for (name, slot), entry in zip(runs, counts):
            mine = [l for l in lines if (l.get("input") == name if run_all else l["stream"] == slot)]
            sc = get(name)
            assert mine and all(("dwell_events" in l) == sc.dwell for l in mine), name
            if not sc.dwell:
                assert all(set(z) == {"entered", "exited"} for z in entry["zones"].values())
                continue
            c = O.Counter(1, 1 << 16)
            c.set_stream(0, *TC._oracle_geometry(sc, config.CLASSES_TO_TRACK))
            d = D.Dwell(c, 1 << 16)
            d.set_dwell(0, True, [z.loiter_frames or 0 for z in sc.zones])
            for l in sorted(mine, key=lambda l: l["frame"]):
                rows = [[tuple(r[:5]) + (config.CLASSES.index(r[5]),) for r in l["tracks"]]]
                c.step(rows)
                d.step(rows)
                want = [{"kind": ("visit", "loiter")[k], "name": sc.zones[z].name, "id": tid, "class": config.CLASSES[cl],
                         "frames": fr} for k, z, tid, cl, fr in d.events[0]]
                assert l["dwell_events"] == want, (name, l["frame"])
                total += len(want)
            for i, z in enumerate(sc.zones):
                for key in ("visits", "frames_total", "frames_max"):
                    arr = getattr(d, key)[0, i]
                    assert entry["zones"][z.name][key] == {config.CLASSES[k]: int(v) for k, v in enumerate(arr) if v}
        assert total > 0
