"""Spectrogram restatement vs the installed scipy (the de-facto pin of the unvendored
dependency, SURVEY.md §8c).  The comparison with the reference itself runs on its stored
outputs (tests/test_oracle_golden.py)."""
import datetime

import numpy as np
import pytest

from oracle import restatement as R
from pyradiotracking_b200 import synth


@pytest.mark.parametrize("nperseg,window", [(256, "hamming"), (1024, "hann"), (64, ("kaiser", 6.0)), (100, "boxcar")])
def test_spectrogram_matches_scipy(nperseg, window):
    scipy_signal = pytest.importorskip("scipy.signal")
    u8 = synth.make_stream(synth.C1, 5, 1)[0][: 2 * 40_000]
    x = R.bytes_to_iq(u8)
    f0, t0, s0 = scipy_signal.spectrogram(x, fs=300000, window=window, nperseg=nperseg, noverlap=0, return_onesided=False)
    f1, t1, s1 = R.spectrogram(x, 300000, window, nperseg)
    assert np.array_equal(f0, f1) and np.array_equal(t0, t1)
    np.testing.assert_allclose(s1, s0, rtol=1e-9)


def test_window_is_scipy_periodic_window():
    sw = pytest.importorskip("scipy.signal")
    for name in ("hamming", "hann", "boxcar"):
        for n in (8, 256, 1000):
            np.testing.assert_array_equal(R.resolve_window(name, n), sw.get_window(name, n))


def test_empty_and_single_column():
    P = R.Params.make()
    f, t, S = R.spectrogram(np.zeros(100, complex), 300000, "hamming", 256)
    assert S.shape == (256, 0) and len(t) == 0
    assert R.extract_runs(P, f, t, S, None, datetime.datetime(2026, 1, 1)) == []
    f, t, S = R.spectrogram(R.bytes_to_iq(synth.make_stream(synth.C1, 0, 1)[0][:512]), 300000, "hamming", 256)
    with pytest.raises(IndexError):       # analyze.py:354 indexes times[1]
        R.extract_sequential(P, f, t, S, None, datetime.datetime(2026, 1, 1))
