"""Line and zone counting on the device (csrc/counting.cu through aicam_counter_*, StreamCounter, the pipeline's
configure_counting and --counting), each compared bit for bit with oracle/counting.py, which keeps its state by track id
where the device keeps it by tracker slot."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from oracle import counting as O
from scenarios import make_scenario

DEV = torch.device("cuda:0")
CLIP = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "aicamera_test_clip.mp4")
gpu = pytest.mark.gpu
NL, NZ, NCLS = 16, 16, 80


def _L():
    from ai_camera_b200 import _lib as L
    return L


def _check(rc):
    _L().check(rc)


def _record(lines, zones):
    """aicam_stream_counting of oracle-shaped geometry."""
    g = _L().StreamCounting()
    g.n_lines, g.n_zones = len(lines), len(zones)
    for i, (a, b, m) in enumerate(lines):
        g.line[i][:] = [a[0], a[1], b[0], b[1]]
        g.line_class_mask[i][:] = list(m)
    for i, (pts, m) in enumerate(zones):
        g.zone_n[i] = len(pts)
        for k, p in enumerate(pts):
            g.zone_xy[i][k][:] = list(p)
        g.zone_class_mask[i][:] = list(m)
    return g


class Counter:
    """A device counter fed with host rows, next to the oracle."""

    def __init__(self, S, T, E):
        from ai_camera_b200.pipeline import StreamCounter
        self.S, self.T, self.E = S, T, E
        self.dev = StreamCounter(DEV, S, T, E)
        self.oracle = O.Counter(S, E)
        i32 = dict(dtype=torch.int32, device=DEV)
        self.out_tracks = torch.zeros((S, T, 6), **i32)
        self.out_count = torch.zeros(S, **i32)
        self.row_slot = torch.zeros((S, T), **i32)
        self.present = torch.ones(S, **i32)

    def set(self, indices, geoms):
        self.dev.set_streams(indices, [_record(*g) for g in geoms])
        for i, g in zip(indices, geoms):
            self.oracle.set_stream(i, *g)

    def set_rc(self, indices, geoms):
        L = _L()
        n = len(indices)
        return L.load().aicam_counter_set_streams(self.dev.handle, (C.c_int32 * n)(*indices),
                                                  (L.StreamCounting * n)(*[_record(*g) for g in geoms]), n, None)

    def step(self, rows, slots, present=None):
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
        self.dev.step(self.out_tracks, self.out_count, C.c_void_p(self.row_slot.data_ptr()),
                      None if present is None else C.c_void_p(self.present.data_ptr()))
        self.oracle.step(rows, present)

    def compare(self, rows, present=None, what=""):
        assert_same(self.dev, self.oracle, rows, present, what)


def assert_same(dev, oracle, rows, present, what):
    torch.cuda.synchronize()
    assert np.array_equal(dev.line_counts.cpu().numpy(), oracle.line_counts), what
    assert np.array_equal(dev.zone_counts.cpu().numpy(), oracle.zone_counts), what
    assert np.array_equal(dev.occupancy.cpu().numpy(), oracle.occupancy), what
    ec, ev, rz = dev.event_count.cpu().numpy(), dev.events.cpu().numpy(), dev.row_zones.cpu().numpy()
    for s in range(len(rows)):
        want = oracle.events[s]
        assert ec[s] == len(want), (what, s)
        assert [tuple(e) for e in ev[s, :ec[s]].tolist()] == want, (what, s)
        if present is None or present[s]:
            assert rz[s, :len(rows[s])].tolist() == oracle.row_zones[s], (what, s)


def _random_geometry(rng, grid, extent, n_lines=NL, n_zones=NZ, n_vert=32):
    def pt():
        return tuple(int(v) for v in rng.integers(-2, extent // grid + 2, 2) * grid)

    def mask():
        return (int(rng.integers(0, 1 << 62)) | 1, int(rng.integers(0, 1 << 16))) if rng.random() < 0.7 else (
            (1 << 64) - 1, (1 << 16) - 1)
    lines = []
    while len(lines) < n_lines:
        a, b = pt(), pt()
        if a != b:
            lines.append((a, b, mask()))
    zones = [([pt() for _ in range(int(rng.integers(3, n_vert + 1)) if n_vert > 3 else 3)], mask()) for _ in range(n_zones)]
    zones[0] = ([pt() for _ in range(n_vert)], mask())  # (at least one zone of the most vertices)
    return lines, zones


class Fleet:
    """Synthetic tracker output: per stream, live tracks in slots, reported or missed, dying and born into free slots
    with new ids; anchors on a coarse grid (ties with lines and vertices), now and then far outside the frame."""

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
                if rng.random() < 0.05:
                    del live[slot]
            free = [k for k in range(self.T) if k not in live]
            rng.shuffle(free)
            for slot in free[:max(0, int(self.T * fill) - len(live))]:
                live[slot] = [self.next_id[s], int(rng.integers(0, self.extent // g)) * g,
                              int(rng.integers(0, self.extent // g)) * g, int(rng.choice([0, 1, 2, 3, 5, 7, 79]))]
                self.next_id[s] += 1
            rep = [k for k in live if rng.random() < 0.7]
            rng.shuffle(rep)
            r = []
            for k in rep:
                t = live[k]
                t[1] += int(rng.integers(-3, 4)) * g
                t[2] += int(rng.integers(-3, 4)) * g
                if rng.random() < 0.1:
                    t[3] = int(rng.choice([0, 2, 79]))
                x, y = t[1], t[2]
                if rng.random() < 0.01:  # far outside: clamped anchors
                    x, y = int(rng.choice([-1, 1])) * (1 << 30), int(rng.choice([-1, 1])) * (1 << 29)
                half = int(rng.integers(0, 30))
                # anchor x = (x1 + x2) / 2 may be a half pixel
                r.append((x - half, y - 40, x + half + int(rng.integers(0, 2)), y, t[0], t[3]))
            rows.append(r)
            slots.append(rep)
        return rows, slots


@gpu
def test_fuzz_at_the_maxima_equals_the_oracle():
    rng = np.random.default_rng(1)
    S, T, E = 64, 256, 256 * 32
    grid, extent = 16, 640
    c = Counter(S, T, E)
    c.set(list(range(S)), [_random_geometry(rng, grid, extent) for _ in range(S)])
    fleet = Fleet(rng, S, T, grid, extent)
    kinds = np.zeros(4, np.int64)
    for t in range(24):
        rows, slots = fleet.step()
        present = (rng.random(S) < 0.8).astype(np.int32) if t % 3 else None
        c.step(rows, slots, present)
        c.compare(rows, present, "step %d" % t)
        for s in range(S):
            for e in c.oracle.events[s]:
                kinds[e[0]] += 1
    assert (kinds > 100).all(), kinds
    assert not c.dev.overflow().any()


def _scenario_geometry():
    all_ = ((1 << 64) - 1, (1 << 16) - 1)
    person_car = (1 | (1 << 2), 0)
    lines = [((960, 0), (960, 1080), all_), ((0, 540), (1920, 540), person_car), ((200, 900), (1700, 100), all_)]
    zones = [([(0, 0), (960, 0), (960, 1080), (0, 1080)], all_),
             ([(300, 200), (1600, 200), (1600, 900), (1000, 900), (1000, 500), (800, 500), (800, 900), (300, 900)], all_),
             ([(100, 100), (1800, 1000), (1800, 100), (100, 1000)], person_car)]
    return lines, zones


@gpu
def test_tracker_driven_counting_equals_the_oracle():
    import gpu_util as G
    S = 4
    scen = [make_scenario(seed=300 + s, n_frames=50, n_objects=14, feat_dim=64, p_miss=0.2) for s in range(S)]
    kmax = max(len(f["boxes"]) for sc in scen for f in sc)
    trk = G.Tracker(S, max_tracks=128, max_dets=kmax, feature_dim=64, stride_k=kmax, n_init=2)
    from ai_camera_b200.pipeline import StreamCounter
    counter = StreamCounter(DEV, S, 128, 4096)
    oracle = O.Counter(S, 4096)
    geo = _scenario_geometry()
    counter.set_streams(list(range(S)), [_record(*geo)] * S)
    for s in range(S):
        oracle.set_stream(s, *geo)
    from ai_camera_b200.pipeline import _DeviceArray
    row_slots = C.c_void_p(_L().load().aicam_tracker_row_slots(trk.h))
    slots_dev = torch.as_tensor(_DeviceArray(trk, row_slots.value, (S, 128), "<i4"), device=DEV)
    slot_of = [{} for _ in range(S)]
    events = 0
    try:
        for t in range(50):
            outs = trk.step([sc[t] for sc in scen])
            counter.step(trk.out_tracks, trk.out_count, row_slots)
            rows = [[tuple(int(v) for v in r) for r in o] for o, _ in outs]
            oracle.step(rows)
            assert_same(counter, oracle, rows, None, "step %d" % t)
            rs = slots_dev.cpu().numpy()
            live = [{int(x[0]) for x in trk.snapshot(s)[0]} for s in range(S)]
            for s in range(S):
                ids = [r[4] for r in rows[s]]
                sl = rs[s, :len(ids)].tolist()
                assert len(set(sl)) == len(sl), (t, s)
                for i, k in zip(ids, sl):
                    assert slot_of[s].setdefault(i, k) == k, (t, s, i)
                slot_of[s] = {i: k for i, k in slot_of[s].items() if i in live[s]}
                events += len(oracle.events[s])
        assert events > 0
    finally:
        trk.close()


# ---- pipeline -------------------------------------------------------------------------------------------------------

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


def _counting(w, h, seed):
    from ai_camera_b200.pipeline import CountingLine, CountingZone, StreamCounting
    rng = np.random.default_rng(seed)
    lines = [CountingLine((w // 2, 0), (w // 2, h), "mid"), CountingLine((0, h // 2), (w, h // 2), classes={"person"})]
    lines += [CountingLine(tuple(int(v) for v in rng.integers(0, w, 2)), tuple(int(v) for v in rng.integers(0, h, 2)))
              for _ in range(3)]
    zones = [CountingZone([(0, 0), (w // 2, 0), (w // 2, h), (0, h)], "left"),
             CountingZone([(w // 4, h // 4), (3 * w // 4, h // 4), (3 * w // 4, 3 * h // 4), (w // 4, 3 * h // 4)], "middle",
                          classes={"person", "car"})]
    return StreamCounting(lines, zones)


def _oracle_geometry(sc, classes):
    from ai_camera_b200 import config
    return ([(x.a, x.b, config.tracked_class_mask(x.classes if x.classes is not None else classes)) for x in sc.lines],
            [(x.points, config.tracked_class_mask(x.classes if x.classes is not None else classes)) for x in sc.zones])


def _host_rows(ot, on, S):
    return [[tuple(int(v) for v in ot[s, k]) for k in range(on[s])] for s in range(S)]


def _video(h, w, seed, n_frames):
    from ai_camera_b200 import synth
    return synth.SynthVideo(1, (h, w), n_frames=n_frames, seed=seed).ring[:, 0]


@gpu
def test_pipeline_counting_equals_the_oracle(blobs, bias):
    """Four streams, two of them counting, one absent at some steps: counters, occupancy, events and row zones equal the
    oracle over the pipeline's own rows; a pipeline without counting launches and returns as before."""
    sizes = [(540, 960), (720, 1280), (540, 960), (480, 640)]
    S, T = len(sizes), 10
    videos = [_video(h, w, 200 + i, T) for i, (h, w) in enumerate(sizes)]
    counting = [_counting(960, 540, 1), None, _counting(960, 540, 2), None]
    pipe = _pipeline(blobs, bias, S, counting=counting)
    plain, neutral = _pipeline(blobs, bias, S), _pipeline(blobs, bias, S, counting=[None] * S)
    assert neutral.counter is None and pipe.counter is not None
    oracle = O.Counter(S, pipe.max_events)
    for s, c in enumerate(counting):
        if c is not None:
            oracle.set_stream(s, *_oracle_geometry(c, pipe.tracker.classes_to_track))
    lib = _L().load()
    launches = {}
    events = 0
    for t in range(T):
        frames = [None if (s == 2 and t in (3, 4)) else videos[s][t] for s in range(S)]
        got = {}
        for name, p in (("pipe", pipe), ("plain", plain), ("neutral", neutral)):
            before = lib.aicam_launch_count()
            got[name] = [x.cpu().numpy() for x in p.step(frames)]
            launches.setdefault(name, set()).add(lib.aicam_launch_count() - before)
        for a, b in zip(got["pipe"], got["plain"]):
            assert np.array_equal(a, b), t
        for a, b in zip(got["neutral"], got["plain"]):
            assert np.array_equal(a, b), t
        present = [f is not None for f in frames]
        rows = _host_rows(got["pipe"][0], got["pipe"][2], S)
        oracle.step(rows, present)
        assert_same(pipe.counter, oracle, rows, present, "step %d" % t)
        events += sum(len(e) for e in oracle.events)
    assert events > 0
    assert launches["plain"] == launches["neutral"] and len(launches["plain"]) == 1
    assert launches["pipe"] == {n + 1 for n in launches["plain"]}
    assert pipe.launches_per_step() == plain.launches_per_step() + 1 == neutral.launches_per_step() + 1
    counts = pipe.counts()
    assert counts[1] == counts[3] == {}
    for s in (0, 2):
        c = counting[s]
        for i, x in enumerate(c.lines):
            assert sum(counts[s]["lines"][x.name]["in"].values()) == oracle.line_counts[s, i, 0].sum()
            assert sum(counts[s]["lines"][x.name]["out"].values()) == oracle.line_counts[s, i, 1].sum()
        for i, x in enumerate(c.zones):
            assert sum(counts[s]["zones"][x.name]["entered"].values()) == oracle.zone_counts[s, i, 0].sum()
            assert sum(counts[s]["zones"][x.name]["occupancy"].values()) == oracle.occupancy[s, i].sum()
    assert not pipe.counter.overflow().any()
    # the stacked step counts too
    stacked = _pipeline(blobs, bias, 2, counting=[counting[0]] * 2)
    oracle = O.Counter(2, stacked.max_events)
    for s in range(2):
        oracle.set_stream(s, *_oracle_geometry(counting[0], stacked.tracker.classes_to_track))
    for t in range(4):
        ot, _, on = [x.cpu().numpy() for x in stacked.step(torch.stack([videos[0][t], videos[2][t]]))]
        rows = _host_rows(ot, on, 2)
        oracle.step(rows)
        assert_same(stacked.counter, oracle, rows, None, "stacked %d" % t)


@gpu
def test_captured_step_follows_presence_and_counting_changes(blobs, bias):
    sizes = [(540, 960), (1080, 1920), (480, 640)]
    S, T = 3, 8
    videos = [_video(h, w, 230 + i, T) for i, (h, w) in enumerate(sizes)]
    masks = [[1, 1, 1], [1, 0, 1], [1, 1, 1], [0, 1, 1], [1, 1, 0], [1, 1, 1], [1, 1, 1], [0, 0, 1]]
    changes = {2: ([1], [_counting(1920, 1080, 5)]), 5: ([0, 2], [None, _counting(640, 480, 6)])}
    start = [_counting(960, 540, 3), None, _counting(640, 480, 4)]
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
    events = 0
    for t in range(T):
        if t in changes:
            for p in (g_pipe, e_pipe):
                p.configure_counting(*changes[t])
        frames = [videos[s][t] if masks[t][s] else None for s in range(S)]
        g_pipe.frame_table.set(frames)
        g.replay()
        e_pipe.step(frames)
        torch.cuda.synchronize()
        for name in ("line_counts", "zone_counts", "occupancy", "event_count", "events", "row_zones"):
            a, b = getattr(g_pipe.counter, name), getattr(e_pipe.counter, name)
            assert torch.equal(a, b), (t, name)
        events += int(e_pipe.counter.event_count.sum())
    assert events > 0
    assert g_pipe.counts() == e_pipe.counts()


@gpu
def test_resets_zero_only_the_selected_streams(blobs, bias):
    from ai_camera_b200.aicamera_tracker import run_batched
    S, T, R = 3, 8, 4
    videos = [_video(540, 960, 260 + i, T) for i in range(S)]
    sc = _counting(960, 540, 7)
    pipe = _pipeline(blobs, bias, S, counting=[sc] * S)
    oracle = O.Counter(S, pipe.max_events)
    for s in range(S):
        oracle.set_stream(s, *_oracle_geometry(sc, pipe.tracker.classes_to_track))
    for t in range(T):
        if t == R:
            pipe.reset_streams([1])
            oracle.reset(1)
            torch.cuda.synchronize()
            assert pipe.counter.line_counts[1].sum() == 0 and pipe.counter.zone_counts[1].sum() == 0
        ot, _, on = [x.cpu().numpy() for x in pipe.step([v[t] for v in videos])]
        rows = _host_rows(ot, on, S)
        oracle.step(rows)
        assert_same(pipe.counter, oracle, rows, None, "step %d" % t)
    # the refill loop: a slot handed to the next source restarts its counts; the other slot keeps counting
    srcs = [[v.cpu().numpy() for v in videos[0]], [v.cpu().numpy() for v in videos[1][:3]]]
    refill = [[v.cpu().numpy() for v in videos[2][:4]]]
    pipe = _pipeline(blobs, bias, 2, counting=[sc] * 2)
    oracle = O.Counter(2, pipe.max_events)
    for s in range(2):
        oracle.set_stream(s, *_oracle_geometry(sc, pipe.tracker.classes_to_track))

    def on_refill(slot, k):
        oracle.reset(slot)

    def on_step(step, batch, table):
        ot, _, on = [x.numpy() for x in table]
        rows = _host_rows(ot, on, 2)
        present = [f is not None for f in batch]
        oracle.step(rows, present)
        assert_same(pipe.counter, oracle, rows, present, "refill step %d" % step)
    run_batched(srcs, pipe, on_step, until="all", refill=iter(refill), on_refill=on_refill)


@gpu
def test_event_overflow_truncates_in_order():
    S, T, E = 3, 32, 5
    c = Counter(S, T, E)
    all_ = ((1 << 64) - 1, (1 << 16) - 1)
    sq = [(0, 0), (100, 0), (100, 100), (0, 100)]
    geo = ([((50, -50), (50, 150), all_)], [(sq, all_)] * 4)
    c.set(list(range(S)), [geo] * S)
    rows = [[(8 - 2, 40, 8 + 2, 50, i + 1, 0) for i in range(n)] for n in (1, 2, 9)]
    slots = [list(range(len(r))) for r in rows]
    c.step(rows, slots)
    c.compare(rows, what="first")
    assert c.dev.overflow().tolist() == [0, 1, 1] and c.oracle.overflow.tolist() == [0, 1, 1]
    rows2 = [[(r[0] + 80, r[1], r[2] + 80, r[3], r[4], r[5]) for r in rr] for rr in rows]  # cross the line, leave nothing
    c.step(rows2, slots)
    c.compare(rows2, what="second")
    assert int(c.dev.line_counts[2].sum()) == 9 and int(c.dev.event_count[2]) == E
    c.dev.reset_streams(torch.tensor([0, 0, 1], dtype=torch.int32, device=DEV))
    assert c.dev.overflow().tolist() == [0, 1, 0] and int(c.dev.zone_counts[2].sum()) == 0


@gpu
def test_abi_rejects_bad_geometry_and_changes_nothing():
    S, T, E = 2, 16, 64
    rng = np.random.default_rng(3)
    a, b = Counter(S, T, E), Counter(S, T, E)
    all_ = ((1 << 64) - 1, (1 << 16) - 1)
    good = _random_geometry(rng, 8, 200, n_lines=3, n_zones=2, n_vert=5)
    for c in (a, b):
        c.set([0, 1], [good, good])
    fleet = Fleet(rng, S, T, 8, 200)
    steps = [fleet.step(0.5) for _ in range(8)]
    for c in (a, b):
        for rows, slots in steps[:4]:
            c.step(rows, slots)
    big = (1 << 20) + 1
    tri = [(0, 0), (5, 0), (0, 5)]
    bad = [([0], [([((0, 0), (0, 0), all_)], [])]),                   # zero-length line
           ([0], [([((0, 0), (big, 0), all_)], [])]),                 # coordinate out of range
           ([0], [([], [([(0, 0), (5, 0)], all_)])]),                 # two vertices
           ([0], [([], [([(0, 0), (5, 0), (0, -big)], all_)])]),
           ([0], [([((0, 0), (1, 0), (0, 1 << 16))], [])]),           # class 80
           ([2], [good]), ([-1], [good]),
           ([1, 0], [good, ([((0, 0), (0, 0), all_)], [])])]          # (the valid first entry is not stored either)
    lib = _L().load()
    torch.cuda.synchronize()
    before = lib.aicam_launch_count()
    for idx, geoms in bad:
        assert b.set_rc(idx, geoms) == -1, idx
    g = _record([((0, 0), (1, 0), all_)] * 3, [(tri, all_)])
    g.n_lines = 17
    assert lib.aicam_counter_set_streams(b.dev.handle, (C.c_int32 * 1)(0), (_L().StreamCounting * 1)(g), 1, None) == -1
    g.n_lines, g.zone_n[0] = 1, 33
    assert lib.aicam_counter_set_streams(b.dev.handle, (C.c_int32 * 1)(0), (_L().StreamCounting * 1)(g), 1, None) == -1
    assert lib.aicam_counter_set_streams(b.dev.handle, None, None, 1, None) == -1
    assert lib.aicam_counter_step(b.dev.handle, None, None, None, None, None) == -1
    assert lib.aicam_launch_count() == before
    for rows, slots in steps[4:]:
        for c in (a, b):
            c.step(rows, slots)
        torch.cuda.synchronize()
        for name in ("line_counts", "zone_counts", "occupancy", "event_count", "events", "row_zones"):
            assert torch.equal(getattr(a.dev, name), getattr(b.dev, name)), name
    b.compare(steps[-1][0], what="after the rejected calls")


def _write_clip(path, frames):
    import cv2
    w = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*"mp4v"), 10, (frames[0].shape[1], frames[0].shape[0]))
    for f in frames:
        w.write(f)
    w.release()
    return str(path)


@gpu
def test_cli_counts_equal_the_oracle_over_its_tracks(blobs, tmp_path):
    import cv2
    from ai_camera_b200 import config, synth, weights
    from ai_camera_b200.aicamera_tracker import load_counting, main, video_frames
    kind, params, tensors = weights.read_blob(blobs[0])
    tensors = dict(tensors)
    for n, b in synth.shifted_class_bias(blobs[0], synth.CLIP_LOGIT_SHIFT).items():
        tensors[n + ".bias"] = b
    yolo = weights.write_blob(str(tmp_path / "yolo_clip.aicw"), kind, params, tensors)
    clip = list(video_frames(CLIP, 12))
    h, w = clip[0].shape[:2]
    paths = [_write_clip(tmp_path / "a.mp4", clip), _write_clip(tmp_path / "b.mp4", [cv2.resize(f, (640, 360)) for f in clip[:8]]),
             _write_clip(tmp_path / "c.mp4", clip[3:10])]
    spec = {"default": {"lines": [{"a": [w // 2, 0], "b": [w // 2, h], "name": "mid"}],
                        "zones": [{"points": [[0, 0], [w // 2, 0], [w // 2, h], [0, h]], "name": "left"}]},
            "b.mp4": {"lines": [{"a": [0, 180], "b": [640, 180]}], "zones": []}}
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
            assert mine and all("events" in l for l in mine)
            sc = get(name)
            o = O.Counter(1, 1 << 16)
            o.set_stream(0, *_oracle_geometry(sc, config.CLASSES_TO_TRACK))
            for l in sorted(mine, key=lambda l: l["frame"]):
                o.step([[tuple(r[:5]) + (config.CLASSES.index(r[5]),) for r in l["tracks"]]])
                want = [{"kind": ("in", "out", "entered", "exited")[k], "name": (sc.lines if k < 2 else sc.zones)[i].name,
                         "id": tid, "class": config.CLASSES[c]} for k, i, tid, c in o.events[0]]
                assert l["events"] == want, (name, l["frame"])
                total += len(want)
            for i, x in enumerate(sc.lines):
                for d, key in ((0, "in"), (1, "out")):
                    assert entry["lines"][x.name][key] == {config.CLASSES[k]: int(v) for k, v in enumerate(o.line_counts[0, i, d]) if v}
            for i, x in enumerate(sc.zones):
                for d, key in ((0, "entered"), (1, "exited")):
                    assert entry["zones"][x.name][key] == {config.CLASSES[k]: int(v) for k, v in enumerate(o.zone_counts[0, i, d]) if v}
        assert total > 0
    # without the flag the track lines carry no events and no counts file is written
    argv = ["--input", paths[0], "--streams", "1", "--output_dir", str(out), "--output_filename", "plain", "--yolo_engine", yolo,
            "--reid_engine", blobs[1]]
    assert main(argv) == 0
    assert all("events" not in json.loads(l) for l in open(out / "plain.tracks.jsonl"))
    assert not (out / "plain.counts.json").exists()
