"""Dwell without a GPU: hand-worked cases pin the rules of oracle/dwell.py (the reference the GPU tests compare
csrc/counting.cu's dwell_kernel against), and the settings types and the --counting loader accept dwell and reject bad
values."""
import json

import pytest

from oracle import counting as O
from oracle import dwell as D

ALL = (0xFFFFFFFFFFFFFFFF, 0xFFFF)
PERSON = (1, 0)
SQUARE = [(0, 0), (10, 0), (10, 10), (0, 10)]
RIGHT = [(10, 0), (20, 0), (20, 10), (10, 10)]


def row_at(x, y, tid, cls=0):
    """A reported row whose bottom-centre anchor is the pixel (x, y)."""
    return (x - 3, y - 20, x + 3, y, tid, cls)


IN, OUT = (5, 5), (50, 50)


class Run:
    """One stream with counting zones and dwell, fed step by step; ``step`` returns (events, row_dwell) of the step."""

    def __init__(self, zones, loiter=(), max_events=64, enabled=True):
        self.c = O.Counter(1, max_events)
        self.c.set_stream(0, [], zones)
        self.d = D.Dwell(self.c, max_events)
        self.d.set_dwell(0, enabled, loiter)

    def step(self, rows):
        """rows: list of rows (None: the stream is absent)."""
        present = None if rows is not None else [0]
        self.c.step([rows or []], present)
        self.d.step([rows or []], present)
        return list(self.d.events[0]), [r[:len(self.c.geometry[0][1])] for r in self.d.row_dwell[0]]

    def at(self, p, tid=1, cls=0):
        return self.step([row_at(*p, tid, cls)])


def test_a_visit_lasts_from_its_entry_report_to_its_first_report_outside():
    r = Run([(SQUARE, ALL)])
    assert r.at(IN) == ([], [[0]])
    assert r.at(IN) == ([], [[1]])
    assert r.at((6, 6)) == ([], [[2]])
    assert r.at(OUT) == ([(D.VISIT, 0, 1, 0, 3)], [[-1]])
    assert r.at(OUT) == ([], [[-1]])
    assert r.d.visits[0, 0, 0] == 1 and r.d.frames_total[0, 0, 0] == 3 and r.d.frames_max[0, 0, 0] == 3
    r.at(IN)
    r.at(OUT)  # a second, shorter visit: the total adds up, the maximum stays
    assert r.d.visits[0, 0, 0] == 2 and r.d.frames_total[0, 0, 0] == 4 and r.d.frames_max[0, 0, 0] == 3


def test_loiter_alert_fires_exactly_at_the_threshold_and_once_per_visit():
    r = Run([(SQUARE, ALL), (RIGHT, ALL)], loiter=[2, 0])
    assert r.at(IN)[0] == []
    assert r.at(IN)[0] == []
    assert r.at(IN) == ([(D.LOITER, 0, 1, 0, 2)], [[2, -1]])   # f - entry == L
    assert r.at(IN)[0] == [] and r.at(IN)[0] == []             # once per visit
    assert r.at((15, 5))[0] == [(D.VISIT, 0, 1, 0, 5)]        # zone 1 (L = 0) never alerts
    assert r.at(IN)[0] == [(D.VISIT, 1, 1, 0, 1)]            # back in zone 0: a new visit there
    assert r.at(IN)[0] == []
    assert r.at(IN)[0] == [(D.LOITER, 0, 1, 0, 2)]            # which alerts again
    assert r.d.visits[0, :2, 0].tolist() == [1, 1]


def test_threshold_one_alerts_at_the_report_after_entry():
    r = Run([(SQUARE, ALL)], loiter=[1])
    assert r.at(IN)[0] == []
    assert r.at(IN)[0] == [(D.LOITER, 0, 1, 0, 1)]


def test_a_class_outside_the_mask_opens_nothing_and_reports_minus_one():
    r = Run([(SQUARE, PERSON)], loiter=[1])
    assert r.at(IN, cls=2) == ([], [[-1]])
    assert r.at(IN, cls=2) == ([], [[-1]])
    assert r.at(OUT, cls=2) == ([], [[-1]])
    assert r.d.visits.sum() == 0


def test_a_class_change_while_a_visit_is_open_leaves_the_visit_as_it_is():
    r = Run([(SQUARE, PERSON)])
    r.at(IN, cls=0)                                   # f = 1: a person enters
    assert r.at(IN, cls=2) == ([], [[-1]])            # now a car inside: state left, -1
    assert r.at(OUT, cls=2) == ([], [[-1]])           # a car outside: still not closed
    assert r.at((7, 7), cls=0) == ([], [[3]])         # a person inside again: the same visit, entry at f = 1
    assert r.at(OUT, cls=0) == ([(D.VISIT, 0, 1, 0, 4)], [[-1]])
    r2 = Run([(SQUARE, PERSON)])
    r2.at(IN, cls=0)
    r2.at(OUT, cls=2)
    assert r2.at(OUT, cls=0)[0] == [(D.VISIT, 0, 1, 0, 2)]  # closes at the person's first report outside


def test_a_track_missed_inside_a_zone_keeps_its_visit_and_its_clock_runs():
    r = Run([(SQUARE, ALL)], loiter=[3])
    r.at(IN)
    assert r.step([]) == ([], [])                     # missed (the stream is present)
    assert r.step([row_at(*OUT, 2)]) == ([], [[-1]])  # missed again, another track reported
    assert r.at(IN) == ([(D.LOITER, 0, 1, 0, 3)], [[3]])
    assert r.step([]) == ([], [])
    assert r.at(OUT)[0] == [(D.VISIT, 0, 1, 0, 5)]


def test_a_new_id_starts_without_visits_and_the_old_open_visit_is_never_counted():
    # on the device the new id is reported from the old track's slot; the previous occupant's visit is dropped
    r = Run([(SQUARE, ALL)])
    r.at(IN, tid=1)
    r.at(IN, tid=1)
    assert r.at(IN, tid=2) == ([], [[0]])
    assert r.at(OUT, tid=2)[0] == [(D.VISIT, 0, 2, 0, 1)]
    assert r.d.visits[0, 0, 0] == 1 and r.d.frames_total[0, 0, 0] == 1


def test_an_absent_step_does_not_advance_the_clock():
    r = Run([(SQUARE, ALL)], loiter=[2])
    r.at(IN)
    assert r.step(None)[0] == []                     # (row_dwell, like row_zones, keeps the last present step's rows)
    assert r.d.clock[0] == 1
    assert r.at(IN) == ([], [[1]])
    assert r.at(IN)[0] == [(D.LOITER, 0, 1, 0, 2)]
    assert r.d.clock[0] == 3


def test_a_reset_and_a_new_geometry_restart_the_state_but_keep_the_settings():
    r = Run([(SQUARE, ALL)], loiter=[2])
    r.at(IN)
    r.at(IN)
    r.at(OUT)
    assert r.d.visits.sum() == 1
    r.at(IN)
    r.c.reset(0)                                      # aicam_counter_reset_streams
    r.d.reset(0)
    assert r.d.visits.sum() == 0 and r.d.clock[0] == 0
    assert r.at(IN) == ([], [[0]])                    # a first report again: the open visit was dropped
    r.at(IN)
    assert r.at(IN)[0] == [(D.LOITER, 0, 1, 0, 2)]    # the threshold is kept
    r.c.set_stream(0, [], [(SQUARE, ALL), (RIGHT, ALL)])  # aicam_counter_set_streams
    r.d.reset(0)
    assert r.d.enabled[0] and r.d.loiter[0][0] == 2
    assert r.at(IN) == ([], [[0, -1]])
    assert r.at(OUT)[0] == [(D.VISIT, 0, 1, 0, 1)]


def test_enabling_mid_stream_treats_tracks_as_first_reports():
    r = Run([(SQUARE, ALL)], loiter=[1], enabled=False)
    r.at(IN)
    assert r.at(IN) == ([], [])                       # disabled: nothing
    assert r.d.clock[0] == 0
    r.d.set_dwell(0, True, [1])
    assert r.at(IN) == ([], [[0]])
    assert r.at(IN)[0] == [(D.LOITER, 0, 1, 0, 1)]
    r.d.set_dwell(0, False, [1])
    r.at(OUT)                                         # disabled while the visit closes: not seen
    r.d.set_dwell(0, True, [1])
    assert r.d.visits.sum() == 0 and r.at(IN) == ([], [[0]])


def test_changing_a_threshold_keeps_the_state_and_never_re_alerts():
    r = Run([(SQUARE, ALL)], loiter=[2])
    for _ in range(3):
        ev = r.at(IN)[0]
    assert ev == [(D.LOITER, 0, 1, 0, 2)]
    r.d.set_dwell(0, True, [4])                       # raised after the alert: the same visit is alerted already
    assert [r.at(IN)[0] for _ in range(4)] == [[]] * 4
    r.at(OUT)
    r.at(IN, tid=2)
    r.at(IN, tid=2)
    r.d.set_dwell(0, True, [1])                       # lowered below the visit's dwell: alerts at its next report
    assert r.at(IN, tid=2) == ([(D.LOITER, 0, 2, 0, 2)], [[2]])


def test_events_are_ordered_by_row_then_zone_and_overflow_keeps_counters():
    zones = [(SQUARE, ALL), (SQUARE, ALL), (SQUARE, ALL)]
    r = Run(zones, loiter=[1, 0, 1], max_events=3)
    r.step([row_at(*IN, 1), row_at(*IN, 2)])
    ev, _ = r.step([row_at(*IN, 1), row_at(*OUT, 2)])
    assert ev == [(D.LOITER, 0, 1, 0, 1), (D.LOITER, 2, 1, 0, 1), (D.VISIT, 0, 2, 0, 1)]
    assert r.d.overflow[0] == 1 and r.d.visits[0, :3, 0].tolist() == [1, 1, 1]
    r.d.reset(0)
    assert r.d.overflow[0] == 0


def test_zones_beyond_the_stream_report_minus_one():
    r = Run([(SQUARE, ALL)])
    r.at(IN)
    assert r.d.row_dwell[0][0] == [1 - 1] + [-1] * 15


# ---- settings types and the command line --------------------------------------------------------------------------------

def test_settings_types():
    from ai_camera_b200.pipeline import CountingZone, StreamCounting
    tri = [(0, 0), (5, 0), (0, 5)]
    assert not StreamCounting([], [CountingZone(tri)]).dwell
    sc = StreamCounting([], [CountingZone(tri), CountingZone(tri, loiter_frames=30, name="door")])
    assert sc.dwell and sc == StreamCounting([], [CountingZone(tri), CountingZone(tri, "door", loiter_frames=30)], dwell=True)
    d = sc.resolve_dwell()
    assert d.enabled == 1 and list(d.loiter_frames) == [0, 30] + [0] * 14
    assert StreamCounting(dwell=True).resolve_dwell().enabled == 1
    assert StreamCounting().resolve_dwell().enabled == 0
    assert CountingZone(tri, loiter_frames=0).loiter_frames == 0 and CountingZone(tri, loiter_frames=1 << 30)
    got = StreamCounting.from_dict({"zones": [{"points": [[0, 0], [5, 0], [0, 5]], "loiter_frames": 90}]})
    assert got.dwell and got.zones[0].loiter_frames == 90
    assert StreamCounting.from_dict({"dwell": True}) == StreamCounting(dwell=True)
    assert StreamCounting.from_dict({"dwell": False}) == StreamCounting()


TRI = [[0, 0], [5, 0], [0, 5]]


@pytest.mark.parametrize("make", [
    lambda P: P.CountingZone(TRI, loiter_frames=-1),
    lambda P: P.CountingZone(TRI, loiter_frames=(1 << 30) + 1),
    lambda P: P.CountingZone(TRI, loiter_frames=2.0),
    lambda P: P.CountingZone(TRI, loiter_frames=True),
    lambda P: P.CountingZone(TRI, loiter_frames="30"),
    lambda P: P.StreamCounting(dwell=1),
    lambda P: P.StreamCounting(dwell="yes"),
    lambda P: P.StreamCounting(dwell=None),
    lambda P: P.StreamCounting.from_dict({"dwell": 1}),
    lambda P: P.StreamCounting.from_dict({"dwell": "true"}),
    lambda P: P.StreamCounting.from_dict({"zones": [{"points": TRI, "loiter_frames": -5}]}),
    lambda P: P.StreamCounting.from_dict({"zones": [{"points": TRI, "loiter_frames": 1.5}]}),
    lambda P: P.StreamCounting.from_dict({"zones": [{"points": TRI, "loiter": 5}]}),
    lambda P: P.StreamCounting.from_dict({"dwel": True}),
])
def test_settings_types_reject_bad_values(make):
    from ai_camera_b200 import pipeline
    with pytest.raises(ValueError):
        make(pipeline)


def test_counting_file_with_dwell(tmp_path):
    from ai_camera_b200.aicamera_tracker import load_counting, parse_arguments
    from ai_camera_b200.pipeline import CountingZone, StreamCounting
    p = tmp_path / "c.json"
    bay = {"points": [[0, 0], [50, 0], [50, 50]], "name": "bay"}
    p.write_text(json.dumps({"default": {"zones": [bay], "dwell": True}, "a.mp4": {"dwell": False},
                             "b.mp4": {"zones": [dict(bay, loiter_frames=45)], "dwell": False}}))
    get = load_counting(str(p))
    zone = CountingZone([(0, 0), (50, 0), (50, 50)], "bay")
    assert get("c.mp4") == StreamCounting([], [zone], dwell=True)
    assert get("a.mp4") == StreamCounting([], [zone])
    assert get("b.mp4").dwell and get("b.mp4").zones[0].loiter_frames == 45  # (a threshold implies dwell)
    for bad in ({"a.mp4": {"dwell": "yes"}}, {"default": {"zones": [dict(bay, loiter_frames=-1)]}}):
        p.write_text(json.dumps(bad))
        with pytest.raises(SystemExit):
            parse_arguments(["--input", "a.mp4", "--streams", "1", "--counting", str(p)])


def test_host_dwell_totals_from_events():
    from ai_camera_b200.aicamera_tracker import CountTotals
    from ai_camera_b200.pipeline import CountingZone, StreamCounting
    tri = [(0, 0), (1, 0), (0, 1)]
    t = CountTotals(StreamCounting([], [CountingZone(tri, "bay")], dwell=True))
    t.add_dwell([{"kind": "visit", "name": "bay", "id": 1, "class": "person", "frames": 7},
                 {"kind": "loiter", "name": "bay", "id": 2, "class": "person", "frames": 9},
                 {"kind": "visit", "name": "bay", "id": 3, "class": "person", "frames": 4},
                 {"kind": "visit", "name": "bay", "id": 4, "class": "car", "frames": 2}])
    assert t.as_dict()["zones"]["bay"] == {"entered": {}, "exited": {}, "visits": {"person": 2, "car": 1},
                                           "frames_total": {"person": 11, "car": 2}, "frames_max": {"person": 7, "car": 2}}
    assert CountTotals(StreamCounting([], [CountingZone(tri, "bay")])).as_dict()["zones"]["bay"] == {"entered": {},
                                                                                                    "exited": {}}
