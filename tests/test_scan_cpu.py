"""Wideband scanner, host half (no GPU): the tone-pair search hbd_scan_detect against the numpy restatement in
scan_ref.detect on seeded random spectra, and the default parameters."""
import ctypes as C

import numpy as np
import pytest

import scan_ref
from habdec_b200 import api


def _psd(rng, case):
    """A float32 PSD with an averaged-noise floor (flat or sloped), planted tone pairs and, in some cases, exact ties."""
    N = int(rng.choice([4096, 5000, 8192, 3000, 1024 + 17]))      # not a multiple of 1024: a short block at the top end
    bw = float(rng.choice([25.0, 38.14697265625, 19.073486328125, 50.0]))
    fs = N * bw
    S = int(rng.choice([1, 2, 8, 64]))
    P = rng.gamma(S, 1.0 / S, N)
    if case % 3 == 1:                                             # sloped floor: 20 dB across the band
        P *= 10.0 ** (2.0 * np.arange(N) / N)
    elif case % 3 == 2:                                           # a step in the floor between blocks
        P[N // 2:] *= 30.0
    n_pairs = int(rng.integers(0, 6))
    for _ in range(n_pairs):
        lo = int(rng.integers(2, N - 80))
        if rng.random() < 0.3:                                    # exactly at a shift limit (bw divides 150 and 1200 for bw = 25, 50)
            d = int(round(rng.choice([150.0, 1200.0]) / bw)) + int(rng.choice([-1, 0, 0, 1]))
        else:
            d = int(rng.integers(2, int(1400 / bw) + 2))
        hi = min(N - 1, lo + max(1, d))
        level = P[lo] * 10.0 ** (rng.uniform(0.5, 3.0))
        P[lo] = level
        P[hi] = level * 10.0 ** (-rng.uniform(0.0, 2.0))           # ratio 0 .. 20 dB: some pairs fail max_tone_ratio_db
        if rng.random() < 0.4:
            P[hi] = P[lo]                                          # equal tones: tie in the visiting order
        if rng.random() < 0.3 and lo + 1 < N:
            P[lo + 1] = P[lo]                                      # equal neighbours: first-maximum rule
        if rng.random() < 0.3:                                     # sidelobes beside the pair
            for k in (lo - d // 2, hi + d // 2):
                if 0 <= k < N:
                    P[k] = level * 0.05
    return P.astype(np.float32), fs


def _params(rng, case):
    if case % 4 == 0:
        return {}
    return dict(min_snr_db=float(rng.choice([6.0, 10.0, 13.0])), min_shift_hz=float(rng.choice([100.0, 150.0, 200.0])),
                max_shift_hz=float(rng.choice([900.0, 1200.0])), max_tone_ratio_db=float(rng.choice([10.0, 15.0, 25.0])))


@pytest.mark.parametrize("seed", range(6))
def test_detect_matches_reference(seed):
    rng = np.random.default_rng(1000 + seed)
    found = 0
    for case in range(50):
        P, fs = _psd(rng, case)
        params = _params(rng, case)
        want = scan_ref.detect(P, fs, **params)
        got = api.scan_detect(P, fs, **params)
        assert [(g["bin_lo"], g["bin_hi"]) for g in got] == [(w[3], w[4]) for w in want], "case %d" % case
        for g, w in zip(got, want):
            for key, v in zip(("center_hz", "shift_hz", "snr_db"), w[:3]):
                assert g[key] == pytest.approx(v, rel=1e-12, abs=1e-300), (case, key)
        found += len(want)
    assert found > 20          # the cases do plant detectable pairs


def test_detect_exact_shift_limits():
    """Pairs exactly min_shift_hz and max_shift_hz apart are found; one bin beyond either limit they are not."""
    N, bw = 8192, 25.0
    fs = N * bw
    for d_bins, ok in ((6, True), (5, False), (48, True), (49, False)):
        P = np.ones(N, dtype=np.float32)
        P[3000] = P[3000 + d_bins] = 1000.0
        got = api.scan_detect(P, fs)
        assert got == [] if not ok else [(s["bin_lo"], s["bin_hi"]) for s in got] == [(3000, 3000 + d_bins)], d_bins
        assert [(s[3], s[4]) for s in scan_ref.detect(P, fs)] == [(s["bin_lo"], s["bin_hi"]) for s in got]


def test_default_params_and_null_params():
    lib = api.load()
    p = api.ScanParams()
    lib.hbd_scan_default_params(C.byref(p))
    assert (p.min_snr_db, p.min_shift_hz, p.max_shift_hz, p.max_tone_ratio_db) == (10.0, 150.0, 1200.0, 15.0)
    assert api.scan_default_params() == scan_ref.DEFAULTS
    rng = np.random.default_rng(5)
    P, fs = _psd(rng, 0)
    P[1000] = P[1020] = 1e3 * P.max()
    out = (api.ScanSignal * 16)()
    n_null = lib.hbd_scan_detect(P.ctypes.data, P.size, fs, None, out, 16)
    n_def = lib.hbd_scan_detect(P.ctypes.data, P.size, fs, C.byref(p), out, 16)
    assert n_null == n_def == len(scan_ref.detect(P, fs)) >= 1


def test_detect_count_beyond_cap_and_argument_errors():
    N, bw = 8192, 25.0
    P = np.ones(N, dtype=np.float32)
    for k in range(5):
        P[500 + 1000 * k] = P[520 + 1000 * k] = 100.0
    lib = api.load()
    out = (api.ScanSignal * 2)()
    assert lib.hbd_scan_detect(P.ctypes.data, N, N * bw, None, out, 2) == 5     # the count, two stored
    assert (out[0].bin_lo, out[1].bin_lo) == (500, 1500)
    assert lib.hbd_scan_detect(P.ctypes.data, N, N * bw, None, None, 0) == 5
    assert lib.hbd_scan_detect(None, N, N * bw, None, None, 0) == api.HBD_ERR_ARG
    assert lib.hbd_scan_detect(P.ctypes.data, 0, N * bw, None, None, 0) == api.HBD_ERR_ARG
    assert lib.hbd_scan_detect(P.ctypes.data, N, 0.0, None, None, 0) == api.HBD_ERR_ARG
    assert lib.hbd_scan_detect(P.ctypes.data, N, N * bw, None, None, 4) == api.HBD_ERR_ARG


def test_reference_welch_definition():
    """scan_ref.welch is the stated definition: a complex exponential on a bin centre lands in that bin of the shifted
    PSD with the window's power gain, and only complete segments count."""
    N, fs = 4096, 4096.0 * 10
    k0 = 1234
    n = np.arange(N * 3 + 100)
    x = np.exp(2j * np.pi * (k0 - N // 2) * n / N)
    P, S = scan_ref.welch(x, N)
    assert S == 5 and int(np.argmax(P)) == k0
    w = scan_ref.window(N)
    assert P[k0] == pytest.approx(np.sum(w) ** 2 / np.sum(w * w), rel=1e-9)
    assert scan_ref.welch(x[:N - 1], N)[1] == 0


def test_binding_returns_every_signal_beyond_its_first_buffer():
    """api.scan_detect asks with room for 16 signals and again with room for all when there are more."""
    N, bw = 65536, 25.0
    P = np.ones(N, dtype=np.float32)
    for k in range(24):
        P[1000 + 2000 * k] = P[1020 + 2000 * k] = 100.0
    got = api.scan_detect(P, N * bw)
    assert len(got) == 24
    assert [(g["bin_lo"], g["bin_hi"]) for g in got] == [(w[3], w[4]) for w in scan_ref.detect(P, N * bw)]
