"""hbd_tracker_reset (host only): a channel handed to a new payload starts with empty telemetry bookkeeping."""
import telemetry_cases as tc
from habdec_b200 import api


def _feed(t, ch, call):
    assert t.push(ch, call, b"1,12:00:00,52.1,21.5,1000", b"AAAA") == 1
    assert t.push(ch, call, b"2,12:00:10,52.3,21.9,9000", b"BBBB") == 1


def test_reset_empties_one_channel_only():
    t = api.Tracker(station=(52.0, 21.0, 100.0), now_unix=tc.CLOCKS[2])
    _feed(t, 3, b"OLD")
    _feed(t, 4, b"KEEP")
    before4 = (t.stats_payload(4), t.get_sentence(4, 1), t.get_sentence(4, 2))
    t.reset(3)
    assert t.stats(3).num_ok_ == 0 and t.stats(3).dist_max_ == 0.0 and t.stats(3).elev_min_ == 90.0
    assert t.get_sentence(3, 1) == b"" and t.get_sentence(3, 2) == b""
    assert t.poll(3) == []
    assert t.stats_payload(3) == api.Tracker(station=(52.0, 21.0, 100.0), now_unix=tc.CLOCKS[2]).stats_payload(3)
    # the other channel keeps its stats, sentences map and unpolled records
    assert (t.stats_payload(4), t.get_sentence(4, 1), t.get_sentence(4, 2)) == before4
    assert t.stats(4).num_ok_ == 2 and [r["frame"] for r in t.poll(4)] == [1, 2]
    # a new payload on the reset channel: frame ids no longer collide with the old payload's
    assert t.push(3, b"NEW", b"2,12:01:00,52.0,21.0,500", b"CCCC") == 1
    assert t.stats(3).num_ok_ == 1 and t.get_sentence(3, 1) == b"" and t.get_sentence(3, 2) == b"NEW,2,12:01:00,52.0,21.0,500*CCCC"
    assert [r["frame"] for r in t.poll(3)] == [2]
    t.reset(99)   # a channel the tracker has never seen: nothing to do
