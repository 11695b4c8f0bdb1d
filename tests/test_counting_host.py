"""Counting without a GPU: the settings types and the --counting loader reject bad values, and hand-worked cases pin the
rules of oracle/counting.py (the reference the GPU tests compare csrc/counting.cu against)."""
import json

import pytest

from oracle import counting as O

ALL = (0xFFFFFFFFFFFFFFFF, 0xFFFF)
PERSON = (1, 0)


def row_at(x, y, tid, cls=0):
    """A reported row whose bottom-centre anchor is the pixel (x, y)."""
    return (x - 3, y - 20, x + 3, y, tid, cls)


def run(steps, lines=(), zones=(), max_events=64):
    """steps: list of row lists of one stream (None: the stream is absent).  Returns (counter, events per step)."""
    c = O.Counter(1, max_events)
    c.set_stream(0, lines, zones)
    out = []
    for rows in steps:
        c.step([rows or []], None if rows is not None else [0])
        out.append(list(c.events[0]))
    return c, out


LINE = [((0, 0), (10, 0), ALL)]  # right-hand side of A->B (y pointing down) is y > 0


@pytest.mark.parametrize("path,want", [
    ([(5, -5), (5, 5)], [O.LINE_IN]),            # left of A->B to its right: in
    ([(5, 5), (5, -5)], [O.LINE_OUT]),
    ([(5, -5), (5, 0), (5, 5)], [O.LINE_IN]),     # on the line: the -1 side, so the crossing is the second move
    ([(5, 5), (5, 0)], [O.LINE_OUT]),
    ([(10, -5), (10, 5)], [O.LINE_IN]),           # through endpoint B
    ([(0, 5), (0, -5)], [O.LINE_OUT]),            # through endpoint A
    ([(9, -1), (11, 1)], [O.LINE_IN]),            # diagonally through B
    ([(11, -5), (11, 5)], []),                    # past the end
    ([(20, -5), (-20, -5)], []),                  # parallel
    ([(-5, 0), (15, 0), (30, 0)], []),            # collinear with the line
    ([(5, -5), (5, 5), (5, -5), (6, 5)], [O.LINE_IN, O.LINE_OUT, O.LINE_IN]),  # every crossing counts
])
def test_line_crossings(path, want):
    _, ev = run([[row_at(x, y, 1)] for x, y in path], lines=LINE)
    got = [e[0] for step in ev for e in step]
    assert got == want
    assert all(e[1:] == (0, 1, 0) for step in ev for e in step)


def test_first_report_never_crosses_and_ids_are_separate():
    _, ev = run([[row_at(5, 5, 1)], [row_at(5, -5, 2)], [row_at(5, 5, 2), row_at(5, -5, 1)]], lines=LINE)
    assert ev == [[], [], [(O.LINE_IN, 0, 2, 0), (O.LINE_OUT, 0, 1, 0)]]


def test_anchor_is_the_doubled_bottom_centre_and_clamps():
    assert O.anchor(1, 2, 4, 9) == (5, 18)
    big = 1 << 30
    assert O.anchor(big, 0, big, -big) == (O.ANCHOR_LIMIT, -O.ANCHOR_LIMIT)
    assert O.anchor(-big, 0, -big, big) == (-O.ANCHOR_LIMIT, O.ANCHOR_LIMIT)
    # a clamped jump still crosses a line near the coordinate limit
    edge = (1 << 20) - 1
    _, ev = run([[(-big, -4, -big, 0, 1, 0)], [(big, -4, big, 0, 1, 0)]], lines=[((edge, -10), (edge, 10), ALL)])
    assert ev == [[], [(O.LINE_OUT, 0, 1, 0)]]


SQUARE = [(0, 0), (10, 0), (10, 10), (0, 10)]
U_SHAPE = [(0, 0), (30, 0), (30, 30), (20, 30), (20, 10), (10, 10), (10, 30), (0, 30)]
BOWTIE = [(0, 0), (10, 10), (10, 0), (0, 10)]


def _in(points, x, y):
    return O.inside([(2 * a, 2 * b) for a, b in points], (2 * x, 2 * y))


@pytest.mark.parametrize("points,x,y,want", [
    (U_SHAPE, 5, 20, True), (U_SHAPE, 25, 20, True), (U_SHAPE, 15, 20, False), (U_SHAPE, 15, 5, True),  # concave
    (BOWTIE, 2, 5, True), (BOWTIE, 8, 5, True), (BOWTIE, 5, 2, False), (BOWTIE, 5, 8, False),          # self-crossing
    # half-open edges: top and left edges belong to the square, bottom and right edges do not; vertices likewise
    (SQUARE, 0, 0, True), (SQUARE, 10, 0, False), (SQUARE, 0, 10, False), (SQUARE, 10, 10, False),
    (SQUARE, 0, 5, True), (SQUARE, 10, 5, False), (SQUARE, 5, 0, True), (SQUARE, 5, 10, False),
    (SQUARE, 5, 5, True), (SQUARE, -1, 5, False),
])
def test_zone_membership(points, x, y, want):
    assert _in(points, x, y) is want
    assert _in(points[::-1], x, y) is want  # (orientation does not matter)


def test_shared_edges_belong_to_one_zone():
    right = [(10, 0), (20, 0), (20, 10), (10, 10)]
    below = [(0, 10), (10, 10), (10, 20), (0, 20)]
    for x, y in [(10, 0), (10, 5), (10, 10), (5, 10), (0, 10), (3, 7)]:
        assert sum(_in(p, x, y) for p in (SQUARE, right, below)) <= 1, (x, y)
    for x, y in [(10, 5), (5, 10)]:  # ((10, 10) belongs to the square below and right of it)
        assert sum(_in(p, x, y) for p in (SQUARE, right, below)) == 1, (x, y)


def test_zone_entries_exits_and_missed_reports():
    zones = [(SQUARE, ALL)]
    c, ev = run([[row_at(5, 5, 1)],        # first report inside: an entry
                 [],                        # missed: keeps its bit
                 [row_at(6, 5, 1)],         # re-reported inside: no new entry
                 None,                      # absent stream: nothing happens
                 [row_at(20, 5, 1)],        # outside: an exit
                 [row_at(5, 5, 1), row_at(7, 7, 2)],
                 []],                       # (track 2 deleted inside: no exit)
                zones=zones)
    assert ev == [[(O.ZONE_ENTRY, 0, 1, 0)], [], [], [], [(O.ZONE_EXIT, 0, 1, 0)],
                  [(O.ZONE_ENTRY, 0, 1, 0), (O.ZONE_ENTRY, 0, 2, 0)], []]
    assert c.zone_counts[0, 0, :, 0].tolist() == [3, 1]
    assert c.occupancy[0, 0, 0] == 0  # rows of the last step
    c.step([[row_at(1, 1, 1), row_at(2, 2, 3, 2), row_at(50, 50, 4)]])
    assert c.occupancy[0, 0, 0] == 1 and c.occupancy[0, 0, 2] == 1 and c.row_zones[0] == [1, 1, 0]


def test_events_are_ordered_by_row_then_lines_then_zones():
    lines = [((0, 0), (10, 0), ALL), ((0, 2), (10, 2), ALL)]
    zones = [([(-50, 1), (50, 1), (50, 50), (-50, 50)], ALL), (SQUARE, ALL)]
    _, ev = run([[row_at(5, -5, 7), row_at(100, 100, 8)], [row_at(5, 5, 7), row_at(5, 5, 8)]], lines, zones)
    assert ev[1] == [(O.LINE_IN, 0, 7, 0), (O.LINE_IN, 1, 7, 0), (O.ZONE_ENTRY, 0, 7, 0), (O.ZONE_ENTRY, 1, 7, 0),
                     (O.ZONE_ENTRY, 0, 8, 0), (O.ZONE_ENTRY, 1, 8, 0)]


def test_class_masks_count_but_membership_is_kept_for_every_row():
    lines = [((0, 0), (10, 0), PERSON)]
    zones = [(SQUARE, PERSON)]
    c, ev = run([[row_at(5, -5, 1, cls=2)],
                 [row_at(5, 5, 1, cls=2)],   # a car crosses and enters: not counted, but its zone bit is kept
                 [row_at(6, 6, 1, cls=0)],   # now a person, still inside: no entry
                 [row_at(6, -5, 1, cls=0)]], # a person leaves and crosses: counted
                lines, zones)
    assert ev == [[], [], [], [(O.LINE_OUT, 0, 1, 0), (O.ZONE_EXIT, 0, 1, 0)]]
    assert c.line_counts[0].sum() == 1 and c.zone_counts[0].sum() == 1
    assert O.class_in((0, 1 << 15), 79) and not O.class_in((0, 1 << 15), 80) and not O.class_in(ALL, -1)


def test_event_overflow_truncates_in_order_and_keeps_counters():
    zones = [(SQUARE, ALL)] * 3
    c, ev = run([[row_at(5, 5, i) for i in range(1, 4)]], zones=zones, max_events=4)
    assert ev[0] == [(O.ZONE_ENTRY, z, i, 0) for i in (1, 2) for z in range(3)][:4]
    assert c.overflow[0] == 1 and c.zone_counts[0, :, 0, 0].tolist()[:3] == [3, 3, 3]
    c.reset(0)
    assert c.overflow[0] == 0 and c.zone_counts.sum() == 0


# ---- settings types and the command line --------------------------------------------------------------------------------

def test_settings_types():
    from ai_camera_b200 import config
    from ai_camera_b200.pipeline import CountingLine, CountingZone, StreamCounting
    sc = StreamCounting([CountingLine((0, 0), (10, 0)), CountingLine([1, 2], [3, 4], name="door", classes=["person"])],
                        [CountingZone([(0, 0), (5, 0), (0, 5)])])
    assert [x.name for x in sc.lines] == ["line0", "door"] and sc.zones[0].name == "zone0"
    assert sc.lines[1].a == (1, 2) and sc.lines[1].classes == {"person"}
    g = sc.resolve({"car"})
    assert (g.n_lines, g.n_zones) == (2, 1)
    assert list(g.line[1]) == [1, 2, 3, 4] and g.zone_n[0] == 3 and list(g.zone_xy[0][1]) == [5, 0]
    assert tuple(g.line_class_mask[0]) == config.tracked_class_mask({"car"})
    assert tuple(g.line_class_mask[1]) == config.tracked_class_mask({"person"})
    d = {"lines": [{"a": [0, 0], "b": [10, 0], "name": "stop"}], "zones": [{"points": [[0, 0], [5, 0], [0, 5]],
                                                                           "classes": ["car", "bus"]}]}
    sc = StreamCounting.from_dict(d)
    assert sc.lines[0].name == "stop" and sc.zones[0].classes == {"car", "bus"} and sc.zones[0].name == "zone0"
    assert StreamCounting.from_dict({}) == StreamCounting()


@pytest.mark.parametrize("make", [
    lambda P: P.CountingLine((0, 0), (0, 0)),
    lambda P: P.CountingLine((0.5, 0), (1, 0)),
    lambda P: P.CountingLine((True, 0), (1, 0)),
    lambda P: P.CountingLine((0, 0, 0), (1, 0)),
    lambda P: P.CountingLine((0, 0), (1 << 20 + 1, 0)),
    lambda P: P.CountingLine((0, 0), (1, 0), classes="person"),
    lambda P: P.CountingLine((0, 0), (1, 0), classes={"unicorn"}),
    lambda P: P.CountingLine((0, 0), (1, 0), name=3),
    lambda P: P.CountingZone([(0, 0), (1, 1)]),
    lambda P: P.CountingZone([(i, i * i) for i in range(33)]),
    lambda P: P.CountingZone([(0, 0), (1, 0), (0, 1.5)]),
    lambda P: P.CountingZone("abc"),
    lambda P: P.StreamCounting([P.CountingLine((0, 0), (1, 0))] * 17),
    lambda P: P.StreamCounting(zones=[P.CountingZone([(0, 0), (1, 0), (0, 1)])] * 17),
    lambda P: P.StreamCounting([P.CountingLine((0, 0), (1, 0), name="a"), P.CountingLine((0, 0), (2, 0), name="a")]),
    lambda P: P.StreamCounting([P.CountingLine((0, 0), (1, 0)), P.CountingLine((0, 0), (2, 0), name="line0")]),
    lambda P: P.StreamCounting([P.CountingZone([(0, 0), (1, 0), (0, 1)])]),
    lambda P: P.StreamCounting.from_dict({"lines": [{"a": [0, 0], "b": [1, 0], "colour": "red"}]}),
    lambda P: P.StreamCounting.from_dict({"gates": []}),
    lambda P: P.StreamCounting.from_dict({"zones": {"points": []}}),
])
def test_settings_types_reject_bad_values(make):
    from ai_camera_b200 import pipeline
    with pytest.raises(ValueError):
        make(pipeline)


def test_counting_file(tmp_path):
    from ai_camera_b200.aicamera_tracker import load_counting, parse_arguments
    from ai_camera_b200.pipeline import CountingLine, CountingZone, StreamCounting
    p = tmp_path / "c.json"
    door = {"a": [0, 100], "b": [200, 100], "name": "door"}
    bay = {"points": [[0, 0], [50, 0], [50, 50]], "name": "bay", "classes": ["car"]}
    p.write_text(json.dumps({"default": {"lines": [door]}, "a.mp4": {"zones": [bay]}, "b.mp4": {"lines": []}}))
    get = load_counting(str(p))
    line = CountingLine((0, 100), (200, 100), name="door")
    assert get("a.mp4") == StreamCounting([line], [CountingZone([(0, 0), (50, 0), (50, 50)], "bay", {"car"})])
    assert get("b.mp4") == StreamCounting()
    assert get("c.mp4") == get(None) == StreamCounting([line])
    args = parse_arguments(["--input", "x/a.mp4", "--streams", "2", "--counting", str(p)])
    assert args.counting_for("a.mp4").zones[0].name == "bay"
    assert parse_arguments(["--input", "a.mp4", "--streams", "2"]).counting_for is None
    for bad in ({"a.mp4": {"lines": [{"a": [0, 0], "b": [0, 0]}]}}, {"a.mp4": {"zones": [{"points": [[0, 0], [1, 1]]}]}},
                {"default": {"lines": [{"a": [0.5, 0], "b": [1, 0]}]}}, {"a.mp4": {"lines": [door, door]}},
                {"a.mp4": []}, ["not", "an", "object"]):
        p.write_text(json.dumps(bad))
        with pytest.raises(SystemExit):
            parse_arguments(["--input", "a.mp4", "--streams", "1", "--counting", str(p)])
    with pytest.raises(SystemExit):  # batched mode only
        parse_arguments(["--input", "a.mp4", "--counting", str(p)])


def test_host_totals_from_events():
    from ai_camera_b200.aicamera_tracker import CountTotals
    from ai_camera_b200.pipeline import CountingLine, CountingZone, StreamCounting
    t = CountTotals(StreamCounting([CountingLine((0, 0), (1, 0), "door")], [CountingZone([(0, 0), (1, 0), (0, 1)], "bay")]))
    t.add([{"kind": "in", "name": "door", "id": 1, "class": "person"}, {"kind": "in", "name": "door", "id": 2, "class": "person"},
           {"kind": "exited", "name": "bay", "id": 2, "class": "car"}])
    assert t.as_dict() == {"lines": {"door": {"in": {"person": 2}, "out": {}}},
                           "zones": {"bay": {"entered": {}, "exited": {"car": 1}}}}
    assert t.panel_lines() == ["door: in 2 out 0", "bay: entered 0 exited 1"]
