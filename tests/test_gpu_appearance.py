"""K8, the tracker's appearance cost, as VALUES on every path that computes it (-m gpu).

    cost[track][det] = min over the track's gallery of max(0, 1 - <g, f>)

One of three kernels computes it, chosen per stream and frame from the tracker's configuration and the frame's
filtered detection count D:

    row kernel     D <= 48, or any D when feature_dim % 32 != 0                      tracker.cu appearance_rows
    TF32x3 kernel  D > 48 when the tracker built it: feature_dim % 32 == 0,           appearance_tf32.cu
                   1 <= nn_budget <= 112 and max_dets > 48
    SGEMM tiling   D > 48, feature_dim % 32 == 0 and no TF32 kernel (nn_budget > 112)  tracker.cu appearance_gemm

Before every frame each value is compared with a float64 reference built from the oracle's raw galleries and with the
oracle's own float32 value, and each case asserts that it reached the code it exists for: the path, the gallery size,
the FIFO wrap, the number of detection tiles.
"""
import math

import numpy as np
import pytest

from scenarios import make_scenario

pytestmark = pytest.mark.gpu

ROW, TF32, SGEMM = "row kernel", "tf32x3", "sgemm"
APP_GEMM_MIN = 48                             # frames with more filtered detections leave the row kernel
TF_N = 112                                    # gallery rows of a TF32 tile: the largest budget it takes
DET_TILE = {ROW: 16, TF32: 128, SGEMM: 64}    # detections per tile of each path
SGEMM_ROWS = 128                              # gallery rows per pass of the SGEMM tiling
BAR = 1e-5                                    # parity bar of the cost (DESIGN section 4)
MARGIN = 2e-5                                 # least distance of a reference value from max_cosine_distance
MAX_COS = 0.2
FRAME_HW = (1080, 1920)


def _long_lived(seed, n_frames, n_objects, feat_dim=512, n_outside=0):
    """Objects that are seen in EVERY frame (tracked class, score >= 0.4), so that the filtered count of each frame is
    exactly n_objects and the galleries grow by one row per frame until the budget, then wrap.  The first n_outside
    objects stand still wholly left of the frame: they are detected, but have no crop and so no feature."""
    rng = np.random.default_rng(seed)
    base = rng.normal(size=(n_objects, feat_dim)).astype(np.float32)
    base /= np.linalg.norm(base, axis=1, keepdims=True)
    cx = rng.uniform(300, 1600, n_objects); cy = rng.uniform(200, 900, n_objects)
    vx = rng.normal(0, 2.0, n_objects); vy = rng.normal(0, 1.0, n_objects)
    h = rng.uniform(80, 200, n_objects); w = h * rng.uniform(0.3, 0.6, n_objects)
    cx[:n_outside], vx[:n_outside], vy[:n_outside] = -w[:n_outside], 0.0, 0.0
    frames = []
    for t in range(n_frames):
        x, y = cx + vx * t + rng.normal(0, 1, n_objects), cy + vy * t + rng.normal(0, 1, n_objects)
        order = rng.permutation(n_objects)
        frames.append(dict(
            boxes=np.stack([x - w / 2, y - h / 2, x + w / 2, y + h / 2], 1).astype(np.float32)[order],
            scores=rng.uniform(0.4, 0.95, n_objects).astype(np.float32)[order],
            classes=np.zeros(n_objects, np.int32),
            feats=(base * rng.uniform(0.5, 2.0, (n_objects, 1)) + 0.05 * rng.normal(size=(n_objects, feat_dim))).astype(np.float32)[order]))
    return frames


def _unit64(x):
    x = np.asarray(x, np.float64)
    return x / np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-7)


def _ref64(ora, f, ids):
    """The cost of every device track (by id) against every filtered detection, in float64 from the raw features the
    oracle holds; inf where the track is not confirmed, its gallery is empty or the detection has no crop."""
    from oracle.tracker import CONFIRMED
    dets = ora._detections(f["boxes"], f["scores"], f["classes"], None, FRAME_HW, f["feats"])
    by_id = {t.track_id: t for t in ora.tracker_core.tracks}
    ref = np.full((len(ids), len(dets)), np.inf)
    cols = [k for k, d in enumerate(dets) if d.feature is not None]
    if cols:
        fd = _unit64([dets[k].feature for k in cols])
        for r, i in enumerate(ids):
            t = by_id[int(i)]
            if t.state == CONFIRMED and t.features:
                ref[r, cols] = np.maximum(0.0, 1.0 - _unit64(t.features) @ fd.T).min(axis=0)
    return ref, len(dets) - len(cols)


def _run_appearance(scenario, n_streams, feature_dim, nn_budget, max_dets, max_tracks=256):
    """scenario: one frame list per stream, all of one length.  Before every frame, the device cost probe against a
    float64 reference and against one oracle DeepSORT per stream; then one step of both, whose returned tuples and
    gallery sizes must be equal.  Returns what the run compared and reached, per path."""
    import gpu_util as G
    from oracle.constants import INFTY_COST
    from oracle.tracker import CONFIRMED, DeepSORT
    assert len(scenario) == n_streams
    tf_built = feature_dim % 32 == 0 and 1 <= nn_budget <= TF_N and max_dets > APP_GEMM_MIN
    stride_k = max(max_dets, max(len(f["boxes"]) for sc in scenario for f in sc))
    paths = {p: dict(n=0, ref=0.0, ora=0.0, tiles=0, no_crop=0) for p in (ROW, TF32, SGEMM)}
    cov = dict(paths=paths, gallery=0, wrap=False, sgemm_passes=0, margin=math.inf, gate_margin=math.inf)
    oras = [DeepSORT(nn_budget=nn_budget) for _ in range(n_streams)]
    trk = G.Tracker(n_streams, max_tracks=max_tracks, max_dets=max_dets, stride_k=stride_k, feature_dim=feature_dim,
                    nn_budget=nn_budget)
    try:
        for t in range(len(scenario[0])):
            frames = [sc[t] for sc in scenario]
            probe = trk.step(frames, probe=True)
            assert trk.probe_launches == (4 if tf_built else 3), (t, trk.probe_launches)
            for s, (f, ora) in enumerate(zip(frames, oras)):
                ids, app, d2 = probe[s]
                wid, wapp, wd2 = ora.probe_costs(f["boxes"], f["scores"], f["classes"], frame_hw=FRAME_HW,
                                                 planted_features=f["feats"])
                where = "frame %d stream %d" % (t, s)
                assert np.array_equal(ids, wid), where
                assert app.shape == wapp.shape, where
                ref, no_crop = _ref64(ora, f, ids)
                nd = app.shape[1]
                path = (ROW if nd <= APP_GEMM_MIN or feature_dim % 32 else TF32 if tf_built else SGEMM)
                rec = paths[path]
                rec["tiles"] = max(rec["tiles"], -(-nd // DET_TILE[path]))
                rec["no_crop"] += no_crop
                if path == SGEMM:
                    ng = max([len(k.features) for k in ora.tracker_core.tracks if k.state == CONFIRMED] + [0])
                    cov["sgemm_passes"] = max(cov["sgemm_passes"], -(-ng // SGEMM_ROWS))
                if not app.size:
                    continue
                fin = np.isfinite(ref)
                assert np.array_equal(app >= INFTY_COST, ~fin), "INFTY_COST pattern differs from float64, " + where
                assert np.array_equal(wapp >= INFTY_COST, ~fin), "INFTY_COST pattern of the oracle, " + where
                assert np.array_equal(d2.view(np.uint32), wd2.view(np.uint32)), "gating distance differs, " + where
                cov["gate_margin"] = min(cov["gate_margin"], float(np.abs(wd2 - 9.487729036781154).min()))
                if fin.any():
                    dref = float(np.abs(app[fin] - ref[fin]).max())
                    dora = float(np.abs(app[fin] - wapp[fin]).max())
                    assert dref <= BAR and dora <= BAR, (path, where, dref, dora)
                    rec["n"] += int(fin.sum())
                    rec["ref"], rec["ora"] = max(rec["ref"], dref), max(rec["ora"], dora)
                    cov["margin"] = min(cov["margin"], float(np.abs(ref[fin] - MAX_COS).min()))
            full = [{k.track_id: k.features[0] for k in o.tracker_core.tracks if len(k.features) == nn_budget} for o in oras]
            outs = trk.step(frames)
            for s, (f, ora) in enumerate(zip(frames, oras)):
                want = ora.update(f["boxes"], f["scores"], f["classes"], frame_hw=FRAME_HW, planted_features=f["feats"])
                assert [tuple(r[:5]) for r in outs[s][0].tolist()] == [w[:5] for w in want], "frame %d stream %d" % (t, s)
                gal = trk.snapshot(s)[0][:, 6]
                assert gal.tolist() == [len(k.features) for k in ora.tracker_core.tracks], "gallery sizes, frame %d" % t
                cov["gallery"] = max(cov["gallery"], int(gal.max(initial=0)))
                cov["wrap"] = cov["wrap"] or any(k.track_id in full[s] and k.features[0] is not full[s][k.track_id]
                                                 for k in ora.tracker_core.tracks)
    finally:
        trk.close()
    for p, r in paths.items():
        if r["n"]:
            print("appearance cost [%s]: %d values, max |diff| from float64 %.2e, from the oracle %.2e, "
                  "%d detection tiles" % (p, r["n"], r["ref"], r["ora"], r["tiles"]))
    print("min margin of float64 to %.1f: %.3e, of d2 to the gate: %.3e; largest gallery %d, wrapped %s" %
          (MAX_COS, cov["margin"], cov["gate_margin"], cov["gallery"], cov["wrap"]))
    assert cov["margin"] > MARGIN, "a value lies within %.0e of max_cosine_distance: choose another seed" % MARGIN
    return cov


def _streams(seed, n_frames, counts, **kw):
    return [_long_lived(seed + s, n_frames, n, **kw) for s, n in enumerate(counts)]


# id -> (scenario, n_streams, feature_dim, nn_budget, max_dets, expected coverage).  Coverage keys: the paths that must
# compare values, the largest gallery, whether a gallery wrapped, the most detection tiles per path, the SGEMM's
# gallery passes and the paths that must see detections without a crop in their frames.
CASES = {
    # row kernel on sparse frames
    "rows_sparse": (lambda: [make_scenario(seed=301, n_frames=40, n_objects=12)], 1, 512, 100, None,
                    dict(paths={ROW})),
    # row kernel on busy frames: 42-48 filtered detections, three full 16-detection tiles
    "rows_busy": (lambda: [make_scenario(seed=302, n_frames=14, n_objects=70, size_range=(25.0, 90.0))], 1, 512, 100,
                  None, dict(paths={ROW}, tiles={ROW: 3})),
    # row kernel, galleries past the budget: the ring wraps at G = 100
    "rows_wrap": (lambda: [_long_lived(303, 125, 5)], 1, 512, 100, None, dict(paths={ROW}, gallery=100, wrap=True)),
    # 1: TF32, all seven 16-column groups, rows 100-111 of the tile masked, FIFO wrap
    "tf32_budget100": (lambda: [_long_lived(401, 110, 60)], 1, 512, 100, 64,
                       dict(paths={TF32}, gallery=100, wrap=True, tiles={TF32: 1})),
    # 2: TF32, wrap at 20, group 1 partly masked
    "tf32_budget20": (lambda: [_long_lived(402, 30, 52)], 1, 512, 20, 64,
                      dict(paths={TF32}, gallery=20, wrap=True, tiles={TF32: 1})),
    # 3: TF32, budget = TF_N: the tile holds only the slot's own rows
    "tf32_budget112": (lambda: [_long_lived(403, 114, 50)], 1, 512, 112, 64,
                       dict(paths={TF32}, gallery=112, wrap=True, tiles={TF32: 1})),
    # 4: TF32 at other feature dims: one K slab; three slabs; the generic gallery-row copy (F % 128 != 0, F > 1024)
    "tf32_f32": (lambda: [_long_lived(404, 30, 56, feat_dim=32)], 1, 32, 100, 64, dict(paths={TF32}, gallery=30)),
    "tf32_f96": (lambda: [_long_lived(405, 30, 56, feat_dim=96)], 1, 96, 100, 64, dict(paths={TF32}, gallery=30)),
    "tf32_f1024": (lambda: [_long_lived(406, 30, 56, feat_dim=1024)], 1, 1024, 100, 64, dict(paths={TF32}, gallery=30)),
    "tf32_f2048": (lambda: [_long_lived(407, 30, 56, feat_dim=2048)], 1, 2048, 100, 64, dict(paths={TF32}, gallery=30)),
    # 5: TF32, two 128-detection tiles (the second partial), galleries of 40 rows
    "tf32_two_tiles": (lambda: [_long_lived(408, 40, 150)], 1, 512, 100, 160,
                       dict(paths={TF32}, gallery=40, tiles={TF32: 2})),
    # 6: TF32, detections without a crop (INFTY_COST columns, empty galleries) inside crowded tiles
    "tf32_no_crop": (lambda: [_long_lived(409, 30, 56, n_outside=6)], 1, 512, 100, 64,
                     dict(paths={TF32}, no_crop={TF32})),
    # 6, 7: SGEMM at the first budget past TF32 eligibility, with detections without a crop
    "sgemm_budget113": (lambda: [_long_lived(410, 30, 56, n_outside=6)], 1, 512, 113, 64,
                        dict(paths={SGEMM}, no_crop={SGEMM}, tiles={SGEMM: 1}, sgemm_passes=1)),
    # 8: SGEMM, second 128-row gallery pass, wrap at 150, second 64-detection tile
    "sgemm_budget150": (lambda: [_long_lived(411, 153, 70, feat_dim=64)], 1, 64, 150, 80,
                        dict(paths={SGEMM}, gallery=150, wrap=True, tiles={SGEMM: 2}, sgemm_passes=2)),
    # 9: row kernel on crowded frames (F % 32 != 0): 53 detections = three full 16-detection tiles and a partial one
    "rows_crowded_f48": (lambda: [_long_lived(412, 24, 53, feat_dim=48)], 1, 48, 100, 64,
                         dict(paths={ROW}, tiles={ROW: 4})),
    # 10: six streams in one handle: 48 -> row kernel, 49 -> TF32; exactly one and just over one 128-detection tile
    "mixed_streams": (lambda: _streams(420, 20, [0, 17, 48, 49, 128, 129]), 6, 512, 100, 129,
                      dict(paths={ROW, TF32}, tiles={ROW: 3, TF32: 2})),
    # 11: max_dets 49: every stream's tile reads the next streams' rows (masked), the last one past the array's end
    "tf32_max_dets49": (lambda: _streams(430, 20, [49, 49, 49]), 3, 512, 100, 49, dict(paths={TF32}, tiles={TF32: 1})),
}


@pytest.mark.parametrize("case", list(CASES))
def test_appearance_cost_and_gate_match_oracle(case):
    """Before every frame, every live track's appearance cost against every filtered detection is within 1e-5 of a
    float64 reference and of the oracle (whose own value goes through a BLAS sgemm), with the same INFTY_COST pattern,
    and the squared Mahalanobis distance equals the oracle's bit for bit; returned tuples are equal every frame."""
    make, n_streams, feature_dim, nn_budget, max_dets, want = CASES[case]
    scenario = make()
    if max_dets is None:
        max_dets = max(8, max(len(f["boxes"]) for f in scenario[0]))
    cov = _run_appearance(scenario, n_streams, feature_dim, nn_budget, max_dets)
    for p in (ROW, TF32, SGEMM):
        assert (cov["paths"][p]["n"] > 0) == (p in want["paths"]), (p, cov["paths"][p]["n"])
    if "gallery" in want:
        assert cov["gallery"] == want["gallery"]
    assert cov["wrap"] == want.get("wrap", False)
    for p, n in want.get("tiles", {}).items():
        assert cov["paths"][p]["tiles"] == n, (p, cov["paths"][p]["tiles"])
    if "sgemm_passes" in want:
        assert cov["sgemm_passes"] == want["sgemm_passes"]
    for p in want.get("no_crop", ()):
        assert cov["paths"][p]["no_crop"] > 0, p


def _smem_optin():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def test_feature_dim_beyond_the_row_kernel_is_rejected():
    """The row kernel stages 16 detection features and 128 minima per block in shared memory; a feature_dim for which
    that exceeds the block's opt-in limit is refused at creation (AICAM_ERR_CAPACITY), not at the first step."""
    import ctypes as C
    import gpu_util as G
    from ai_camera_b200._lib import TrackerConfig
    f_max = (_smem_optin() // 4 - 8 * 16) // 16
    for F in (f_max + 1, 4096):
        cfg = TrackerConfig(1, 4, 8, F, 0.2, 0.7, 70, 3, 4, 0)
        h = C.c_void_p()
        rc = G.lib().aicam_tracker_create(C.byref(cfg), C.byref(h))
        if rc == 0:
            G.lib().aicam_tracker_destroy(h)
        assert rc == -4, (F, rc)
        assert b"feature_dim" in G.lib().aicam_last_error(), F


def test_largest_feature_dim_matches_oracle():
    """At the largest accepted feature_dim the row kernel uses all the shared memory a block can have: costs, gating
    and returned tuples equal the oracle's on a small tracker."""
    f_max = (_smem_optin() // 4 - 8 * 16) // 16
    cov = _run_appearance([_long_lived(440, 5, 2, feat_dim=f_max)], 1, f_max, 4, 8, max_tracks=4)
    assert cov["paths"][ROW]["n"] > 0 and cov["gallery"] == 4
