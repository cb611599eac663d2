"""Cross-device matcher (SURVEY.md section 8f rank 1): native loop (include/rt_matcher.h, host code -- no GPU needed)
vs the oracle restatement vs fixtures produced by the UNMODIFIED reference (oracle/make_matcher_golden.py)."""
import datetime
import json
import os

import numpy as np
import pytest

from oracle import matcher as M
from pyradiotracking_b200 import messages
from pyradiotracking_b200.match import SignalMatcher

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _golden(name):
    with open(os.path.join(GOLDEN, f"matcher_{name}.json")) as f:
        return json.load(f)


class _Q:
    def __init__(self):
        self.items = []

    def put(self, x):
        self.items.append(x)


def _as_signals(sigs):
    out = []
    for s in sigs:
        r = messages.Signal(s.device, s.ts, s.frequency, s.duration, s.avg + 3.0, s.avg, 1.0, -95.0, 10.0)
        r.idx = s.idx
        out.append(r)
    return out


def _run_oracle(name):
    o = M.OracleMatcher(**M.matcher_kwargs(name))
    for s in M.make_signals(name):
        o.add(s)
    return o


@pytest.mark.parametrize("name", list(M.CASES))
def test_oracle_matches_reference_fixture(name):
    g = _golden(name)
    assert g["kwargs"] == M.matcher_kwargs(name) and g["n_signals"] == len(M.make_signals(name))
    o = _run_oracle(name)
    assert M.groups_as_ids(o.emitted) == g["emitted"]
    assert M.groups_as_ids(o._matched) == g["open"]
    for grp, view in zip(o.emitted, g["views"]):
        assert grp.ts.isoformat() == view["ts"] and grp.frequency == view["frequency"]
        assert grp.duration // datetime.timedelta(microseconds=1) == view["duration_us"]


@pytest.mark.parametrize("name", list(M.CASES))
@pytest.mark.parametrize("chunk", [1, 7, 10 ** 9])
def test_native_matcher_matches_reference_fixture(name, chunk):
    """One Signal per call (the reference's consumer loop), small batches, one batch: identical queue content."""
    g = _golden(name)
    q = _Q()
    m = SignalMatcher(signal_queue=q, **M.matcher_kwargs(name))
    sigs = _as_signals(M.make_signals(name))
    for i in range(0, len(sigs), chunk):
        if chunk == 1:
            m.add(sigs[i])
        else:
            m.add_batch(sigs[i:i + chunk])
    assert M.groups_as_ids(q.items) == g["emitted"]
    assert M.groups_as_ids(m._matched) == g["open"]
    for grp, view in zip(q.items, g["views"]):          # the reference's derived views of a group
        assert grp.ts.isoformat() == view["ts"] and grp.frequency == view["frequency"]
        assert grp.duration // datetime.timedelta(microseconds=1) == view["duration_us"]
        assert grp._avgs == view["avgs"]
        assert grp.as_list[:3] == [grp.ts, grp.frequency, grp.duration] and grp.header[3:] == m.devices
    m.close()


def test_native_matcher_equals_oracle_on_random_long_sequences():
    rng = np.random.default_rng(99)
    for trial in range(6):
        n_dev = int(rng.integers(2, 9))
        kw = dict(device=[str(d) for d in range(n_dev)], matching_timeout_s=float(rng.choice([0.01, 0.1, 2.0])),
                  matching_time_diff_s=float(rng.choice([0.0, 0.0005, 0.003])), matching_bandwidth_hz=float(rng.choice([0.0, 1000.0, 5000.0])),
                  matching_duration_diff_ms=[None, 0.0, 0.0015, 2.0, 7.001][int(rng.integers(5))])
        sigs = []
        t = 0
        for k in range(5000):
            t += int(rng.exponential(400))
            sigs.append(M.Sig(str(int(rng.integers(n_dev))), M.T0 + datetime.timedelta(microseconds=t + int(rng.integers(-3000, 3000))),
                              150e6 + float(rng.integers(-3, 4)) * 1000.0, datetime.timedelta(microseconds=int(rng.integers(8, 41)) * 1000 + int(rng.integers(-2, 3))),
                              float(rng.normal(-60, 5)), k))
        o = M.OracleMatcher(**kw)
        for s in sigs:
            o.add(s)
        q = _Q()
        m = SignalMatcher(signal_queue=q, **kw)
        m.add_batch(_as_signals(sigs))
        assert M.groups_as_ids(q.items) == M.groups_as_ids(o.emitted), kw
        assert M.groups_as_ids(m._matched) == M.groups_as_ids(o._matched), kw
        m.close()


def test_non_signal_messages_are_ignored_and_naive_timestamps_work():
    q = _Q()
    m = SignalMatcher(["0", "1"], 1.0, 0.0, 0.0, q)
    m.add(messages.StateMessage("0", datetime.datetime(2026, 1, 1), 1))
    assert m._matched == [] and q.items == []
    t = datetime.datetime(2026, 1, 1, 0, 0, 0)
    a = messages.Signal("0", t, 150e6, datetime.timedelta(milliseconds=10), -50, -55, 1, -90, 30)
    b = messages.Signal("1", t + datetime.timedelta(milliseconds=5), 150e6, datetime.timedelta(milliseconds=10), -50, -57, 1, -90, 30)
    c = messages.Signal("0", t + datetime.timedelta(seconds=3), 150e6, datetime.timedelta(milliseconds=10), -50, -57, 1, -90, 30)
    m.add(a), m.add(b)
    assert [sorted(g._sigs) for g in m._matched] == [["0", "1"]]
    m.add(c)                                            # 3 s later: the first group times out and is published
    assert len(q.items) == 1 and q.items[0]._avgs == [-55.0, -57.0] and q.items[0].ts == t
    assert q.items[0].duration == datetime.timedelta(milliseconds=10)
    m.close()
