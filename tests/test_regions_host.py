"""Per-stream include and exclude regions, host side: the rule as oracle/regions.py states it (the device's region test
is compared with it in test_gpu_regions.py), StreamSettings' region fields and the --stream_settings file."""
import json

import numpy as np
import pytest

from oracle import regions as R

SQUARE = [(0, 0), (10, 0), (10, 10), (0, 10)]
U_SHAPE = [(0, 0), (30, 0), (30, 30), (20, 30), (20, 10), (10, 10), (10, 30), (0, 30)]
BOWTIE = [(0, 0), (10, 10), (10, 0), (0, 10)]
F32 = np.float32


def box_at(x, y):
    """A box whose doubled anchor is (2x, 2y) exactly."""
    return (x - 3, y - 8, x + 3, y)


def keeps(includes, excludes, box):
    return R.keep((includes, excludes), box)


@pytest.mark.parametrize("x,y,want", [
    # half-open: the top and left edges and the top-left vertex belong to the square, the others do not
    (0, 0, True), (10, 0, False), (0, 10, False), (10, 10, False),
    (0, 5, True), (10, 5, False), (5, 0, True), (5, 10, False), (5, 5, True), (-1, 5, False),
])
def test_anchor_on_edges_and_vertices(x, y, want):
    assert keeps([SQUARE], [], box_at(x, y)) is want
    assert keeps([], [SQUARE], box_at(x, y)) is (not want)


def test_anchor_is_the_doubled_bottom_centre_on_the_grid():
    assert R.anchor(1.0, 2.0, 4.0, 7.0) == (5, 14)
    assert R.anchor(0.25, 0.0, 0.5, 3.75) == (0, 7)       # floor(0.75), floor(7.5)
    assert R.anchor(-0.5, 0.0, 0.25, -0.25) == (-1, -1)   # floor rounds down, also below zero
    big = float(1 << 25)
    assert R.anchor(big, 0, big, -big) == (1 << 24, -(1 << 24))


def test_float32_sum_rounds_across_an_integer():
    x1 = np.nextafter(F32(1), F32(0))  # 0.99999994
    assert float(x1) + 19.0 < 20.0     # in exact arithmetic the sum is below 20 ...
    assert R.anchor(x1, 0, 19.0, 5.0) == (20, 10)  # ... in float32 it rounds to 20: on the square's right edge
    assert not keeps([SQUARE], [], (x1, 0, 19.0, 5.0))
    assert keeps([SQUARE], [], (0.5, 0, 19.0, 5.0))  # 19.5 -> 19: inside


def test_twice_y2_just_below_an_integer():
    y2 = np.nextafter(F32(10), F32(0))  # 2 * y2 = 19.999998 exactly
    assert R.anchor(4.0, 0, 6.0, y2) == (10, 19)
    assert keeps([SQUARE], [], (4.0, 0, 6.0, y2))
    assert not keeps([SQUARE], [], (4.0, 0, 6.0, 10.0))


@pytest.mark.parametrize("points,x,y,want", [
    (U_SHAPE, 5, 20, True), (U_SHAPE, 25, 20, True), (U_SHAPE, 15, 20, False), (U_SHAPE, 15, 5, True),  # concave
    (BOWTIE, 2, 5, True), (BOWTIE, 8, 5, True), (BOWTIE, 5, 2, False), (BOWTIE, 5, 8, False),          # self-crossing
])
def test_concave_and_self_intersecting_polygons(points, x, y, want):
    assert keeps([points], [], box_at(x, y)) is want
    assert keeps([points[::-1]], [], box_at(x, y)) is want


def test_overlapping_includes_and_exclude_wins():
    other = [(5, 5), (15, 5), (15, 15), (5, 15)]
    for x, y in [(7, 7), (2, 2), (12, 12)]:  # in both, in the first only, in the second only
        assert keeps([SQUARE, other], [], box_at(x, y))
    assert not keeps([SQUARE, other], [], box_at(20, 20))
    hole = [(6, 6), (9, 6), (9, 9), (6, 9)]
    assert not keeps([SQUARE, other], [hole], box_at(7, 7))
    assert keeps([SQUARE, other], [hole], box_at(2, 2))
    assert not keeps([SQUARE], [SQUARE], box_at(5, 5))  # inside an include and an exclude: dropped


def test_no_include_means_the_whole_frame():
    for x, y in [(-(1 << 20), 3), (15, 20), (1 << 20, 1 << 20)]:  # ((15, 20): in the U's notch)
        assert keeps([], [], box_at(x, y))
        assert keeps([], [U_SHAPE], box_at(x, y))
    assert not keeps([], [U_SHAPE], box_at(5, 20))
    assert R.keep_mask(([], []), np.zeros((3, 4), F32)).tolist() == [True] * 3


def test_compaction_keeps_scan_order():
    boxes = np.array([box_at(5, 5), box_at(50, 5), box_at(2, 2), box_at(7, 1), box_at(9, 9)], F32)
    scores = np.array([0.9, 0.8, 0.7, 0.6, 0.5], F32)
    labels = np.array([0, 2, 0, 7, 0], np.int32)
    n, b, s, l = R.compact(([SQUARE], [[(6, 0), (8, 0), (8, 2), (6, 2)]]), 5, boxes, scores, labels)
    assert n == 3
    assert b[:3].tolist() == boxes[[0, 2, 4]].tolist() and not b[3:].any()
    assert s.tolist() == [F32(0.9), F32(0.7), F32(0.5), 0, 0] and l.tolist() == [0, 0, 0, 0, 0]
    n, *_ = R.compact(([SQUARE], []), 2, boxes, scores, labels)  # rows past num_dets are not detections
    assert n == 1


# ---- StreamSettings ---------------------------------------------------------------------------------------------------

def test_settings_carry_and_resolve_regions():
    from ai_camera_b200.pipeline import StreamSettings
    st = StreamSettings(include_regions=[[[0, 0], [100, 0], [100, 50]]], exclude_regions=(SQUARE, U_SHAPE))
    assert st.include_regions == (((0, 0), (100, 0), (100, 50)),)
    assert st.exclude_regions == (tuple(SQUARE), tuple(U_SHAPE))
    assert st.has_regions() and not StreamSettings().has_regions()
    assert len(st.resolve()) == 2
    r = st.resolve_region()
    assert r.n_polygons == 3 and list(r.kind)[:3] == [0, 1, 1] and list(r.n_vertices)[:3] == [3, 4, 8]
    assert [tuple(r.xy[2][k]) for k in range(8)] == U_SHAPE
    assert StreamSettings().resolve_region().n_polygons == 0
    assert StreamSettings.from_dict({"exclude_regions": [SQUARE]}) == StreamSettings(exclude_regions=[SQUARE])
    eight = StreamSettings(include_regions=[SQUARE] * 5, exclude_regions=[BOWTIE] * 3)
    assert eight.resolve_region().n_polygons == 8
    limit = 1 << 20
    StreamSettings(include_regions=[[(-limit, -limit), (limit, -limit), (limit, limit)] + [(0, 0)] * 29])


@pytest.mark.parametrize("kw", [
    dict(include_regions=[[(0, 0), (1.5, 0), (1, 1)]]),                        # not an integer
    dict(include_regions=[[(0, 0), (True, 0), (1, 1)]]),
    dict(exclude_regions=[[(0, 0), ((1 << 20) + 1, 0), (1, 1)]]),              # beyond 2^20
    dict(include_regions=[[(0, 0), (1, 0)]]),                                  # 2 vertices
    dict(include_regions=[[(k, k * k) for k in range(33)]]),                   # 33 vertices
    dict(include_regions=[SQUARE] * 5, exclude_regions=[SQUARE] * 4),          # 9 polygons in total
    dict(include_regions=[SQUARE] * 9),
    dict(include_regions="[[0, 0], [1, 0], [1, 1]]"),                          # a string
    dict(include_regions=["abc"]),
    dict(exclude_regions=[[(0, 0), (1, 0), (1, 1, 1)]]),
    dict(exclude_regions=[[(0, 0), (1, 0), "xy"]]),
    dict(include_regions=None),
])
def test_settings_reject_bad_regions(kw):
    from ai_camera_b200.pipeline import StreamSettings
    with pytest.raises(ValueError):
        StreamSettings(**kw)


def test_from_dict_rejects_unknown_keys():
    from ai_camera_b200.pipeline import StreamSettings
    with pytest.raises(ValueError):
        StreamSettings.from_dict({"include_region": [SQUARE]})


def test_stream_settings_file_with_regions(tmp_path):
    from ai_camera_b200.aicamera_tracker import load_stream_settings, parse_arguments
    from ai_camera_b200.pipeline import StreamSettings
    p = tmp_path / "s.json"
    spec = {"default": {"exclude_regions": [[[0, 0], [1920, 0], [1920, 360], [0, 360]]]},
            "door.mp4": {"include_regions": [[[100, 400], [900, 400], [900, 1080], [100, 1080]]], "exclude_regions": []}}
    p.write_text(json.dumps(spec))
    get = load_stream_settings(str(p), 0.25)
    assert get("door.mp4") == StreamSettings(conf_threshold=0.25, include_regions=[[(100, 400), (900, 400), (900, 1080),
                                                                                  (100, 1080)]])
    assert get("other.mp4").exclude_regions == (((0, 0), (1920, 0), (1920, 360), (0, 360)),)
    args = parse_arguments(["--input", "door.mp4", "--streams", "1", "--stream_settings", str(p)])
    assert args.settings_for("door.mp4").has_regions()
    for bad in ({"a.mp4": {"include_regions": [[[0, 0], [1, 0]]]}}, {"a.mp4": {"exclude_regions": "everywhere"}},
                {"a.mp4": {"include_regions": [[[0, 0], [0.5, 0], [1, 1]]]}},
                {"a.mp4": {"include_regions": [[[0, 0], [1 << 21, 0], [1, 1]]]}},
                {"default": {"include_regions": [[[0, 0], [9, 0], [9, 9]]] * 9}}, {"a.mp4": {"regions": []}}):
        p.write_text(json.dumps(bad))
        with pytest.raises(SystemExit):
            parse_arguments(["--input", "a.mp4", "--streams", "1", "--stream_settings", str(p)])
