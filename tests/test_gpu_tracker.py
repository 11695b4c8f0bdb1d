"""Device DeepSORT association vs the oracle and the reference-recorded golden fixtures (-m gpu)."""
import numpy as np
import pytest

from golden_util import assert_same_tracking, load, run_oracle, scenario_digest
from scenarios import GOLDEN_SCENARIOS, GOLDEN_TRACKER_KW, make_scenario

pytestmark = pytest.mark.gpu


def _lsap_cases(rng, n, shapes):
    for t in range(n):
        nr, nc = shapes(rng)
        kind = t % 4
        if kind == 0:
            c = rng.random((nr, nc))
        elif kind == 1:
            c = rng.integers(0, 4, (nr, nc)).astype(np.float64)
        elif kind == 2:
            c = rng.random((nr, nc))
            c[c > 0.2] = 0.20001
        else:
            c = rng.random((nr, nc))
            c[rng.random((nr, nc)) < 0.5] = 0.70001
        yield c.astype(np.float32)


def test_lsap_matches_scipy_small_shapes():
    """Bit-identical assignments, ties included (SURVEY Appendix B)."""
    import gpu_util as G
    from scipy.optimize import linear_sum_assignment
    rng = np.random.default_rng(7)
    for nr in range(1, 14):
        for nc in range(1, 14):
            costs = np.stack(list(_lsap_cases(rng, 24, lambda r: (nr, nc))))
            got = G.lsap(costs)
            for c, g in zip(costs, got):
                want = np.full(nr, -1)
                r, cc = linear_sum_assignment(c)
                want[r] = cc
                assert np.array_equal(g, want), (nr, nc, c.tolist())


@pytest.mark.parametrize("shape", [(40, 40), (33, 70), (70, 33), (128, 100), (300, 300)], ids=str)
def test_lsap_matches_scipy_large(shape):
    import gpu_util as G
    from scipy.optimize import linear_sum_assignment
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    costs = np.stack(list(_lsap_cases(rng, 8, lambda r: shape)))
    got = G.lsap(costs)
    for c, g in zip(costs, got):
        want = np.full(shape[0], -1)
        r, cc = linear_sum_assignment(c)
        want[r] = cc
        assert np.array_equal(g, want)


def test_gating_matches_reference_golden():
    import gpu_util as G
    g = load("kalman.npz")
    for n in sorted(set(g["gate_n"].tolist())):
        sel = g["gate_n"] == n
        got = G.kf_gating(g["gate_in"][sel], g["gate_z"][sel][:, :n])
        assert np.array_equal(got.view(np.uint32), g["gate_out"][sel][:, :n].view(np.uint32)), n


@pytest.mark.parametrize("name", sorted(GOLDEN_SCENARIOS))
def test_tracker_matches_reference_golden(name):
    """Ids, lifecycle counters, returned tuples and the fp32 Kalman state of every live track after
    every frame equal what the real reference produced."""
    import gpu_util as G
    kw = GOLDEN_SCENARIOS[name]
    frames = make_scenario(**kw)
    want = load("tracker_%s.npz" % name)
    assert scenario_digest(frames) == bytes(want["digest"]).decode()
    got = G.run_gpu_tracker(frames, feature_dim=kw.get("feat_dim", 512), **GOLDEN_TRACKER_KW.get(name, {}))
    assert_same_tracking(got, want, name)


@pytest.mark.parametrize("seed,n_objects,n_frames", [(101, 16, 60), (102, 60, 30), (103, 150, 12)])
def test_tracker_matches_oracle_fresh_seeds(seed, n_objects, n_frames):
    import gpu_util as G
    frames = make_scenario(seed=seed, n_frames=n_frames, n_objects=n_objects, size_range=(30.0, 150.0))
    assert_same_tracking(G.run_gpu_tracker(frames), run_oracle(frames), "seed %d" % seed)


def test_tracker_crowded_scene_300_persons():
    """BASELINE config 5: 300 persons per frame (ReID batch 300, 300 x 300 association per stream); ids,
    lifecycle and Kalman state bit-exact against the oracle, gallery growing over the frames."""
    import gpu_util as G
    frames = make_scenario(seed=104, n_frames=10, n_objects=300, size_range=(20.0, 90.0))
    got = G.run_gpu_tracker(frames, max_tracks=512)
    assert_same_tracking(got, run_oracle(frames), "crowded 300")
    assert got["trk_off"][-1] - got["trk_off"][-2] >= 150  # a crowded scene: hundreds of live tracks per frame


def test_tracker_streams_are_independent():
    """Several streams in one handle give what separate single-stream trackers give."""
    import gpu_util as G
    scen = [make_scenario(seed=200 + s, n_frames=20, n_objects=4 + 3 * s) for s in range(5)]
    kmax = max(len(f["boxes"]) for sc in scen for f in sc)
    trk = G.Tracker(5, max_tracks=128, max_dets=kmax, stride_k=kmax)
    multi = [[] for _ in scen]
    try:
        for t in range(20):
            for s, (o, c) in enumerate(trk.step([sc[t] for sc in scen])):
                multi[s].append(o)
    finally:
        trk.close()
    for s, sc in enumerate(scen):
        single = run_oracle(sc)
        for t in range(20):
            assert np.array_equal(multi[s][t], single["out"][single["out_off"][t]:single["out_off"][t + 1]])


def test_tracker_empty_frames_and_capacity_flag():
    import gpu_util as G
    trk = G.Tracker(1, max_tracks=4, max_dets=8, stride_k=8, feature_dim=16, n_init=2, max_age=1)
    try:
        e = dict(boxes=np.zeros((0, 4), np.float32), scores=np.zeros(0, np.float32), classes=np.zeros(0, np.int32),
                 feats=np.zeros((0, 16), np.float32))
        assert len(trk.step([e])[0][0]) == 0
        six = dict(boxes=np.asarray([[100 * i, 50, 100 * i + 40, 150] for i in range(6)], np.float32),
                   scores=np.full(6, 0.9, np.float32), classes=np.zeros(6, np.int32),
                   feats=np.eye(6, 16, dtype=np.float32))
        trk.step([six])
        assert trk.overflow()[0] & 1  # only 4 track slots
        assert len(trk.snapshot(0)[0]) == 4
    finally:
        trk.close()


def test_tracker_without_features_matches_reference_semantics():
    """feats == NULL: every appearance cost is INFTY_COST and the galleries stay as they were (the reference with
    every Detection.feature None); the same frames through the oracle with all crops invalid."""
    import gpu_util as G
    import torch
    from oracle.tracker import DeepSORT
    frames = make_scenario(seed=41, n_frames=25, n_objects=6, feat_dim=32, p_miss=0.0, p_fp=0.0)
    kmax = max(8, max(len(f["boxes"]) for f in frames))
    trk = G.Tracker(1, max_tracks=64, max_dets=kmax, stride_k=kmax, feature_dim=32)
    ora = DeepSORT(reid_fn=lambda frame, rects: np.zeros((0, 32), np.float32))  # wrong row count -> no features (:174-178)
    try:
        for t, f in enumerate(frames):
            # poison the scratch buffers a feature-less step must not read
            trk.feats.fill_(float("nan"))
            got = trk.step([f], feats_null=True)[0][0]
            want = ora.update(f["boxes"], f["scores"], f["classes"], frame_bgr=np.zeros((1080, 1920, 3), np.uint8))
            assert [tuple(r[:5]) for r in got.tolist()] == [w[:5] for w in want], t
            ints, _ = trk.snapshot(0)
            assert (ints[:, 6] == 0).all()  # no gallery ever grows
    finally:
        trk.close()
