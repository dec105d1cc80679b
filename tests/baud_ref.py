"""numpy restatement of the baud-rate estimator stated in include/habdec_b200.h (steps 1-5), for the GPU's histograms and
estimates to be compared with bit for bit.  Input: a channel's discriminator output in stream order since the estimator
(re)started."""
import math

import numpy as np

CANDIDATES = (50, 75, 100, 150, 200, 300, 600)


def geometry(fs: float):
    """(Lmax, m): histogram length and debounce at fs_dec = fs."""
    return int(math.ceil(6.5 * fs / 50)), max(1, int(math.floor(fs / 2400)))


def edges(d, m: int) -> np.ndarray:
    """Steps 1-2: positions of the accepted edges.  Walked over the runs of equal sign: a streak of the opposite sign is a
    whole run (the next run has the current sign again), so an edge is an opposite-sign run of at least m samples."""
    s = np.asarray(d, dtype=np.float32) > 0
    if not s.size:
        return np.zeros(0, dtype=np.int64)
    starts = np.concatenate(([0], np.flatnonzero(s[1:] != s[:-1]) + 1))
    lengths = np.diff(np.concatenate((starts, [s.size])))
    cur = bool(s[0])
    out = []
    for st, ln, v in zip(starts.tolist(), lengths.tolist(), s[starts].tolist()):
        if v != cur and ln >= m:
            out.append(st)
            cur = v
    return np.asarray(out, dtype=np.int64)


def edges_literal(d, m: int) -> np.ndarray:
    """Steps 1-2 sample by sample, as the text states them (slow; checks edges())."""
    s = np.asarray(d, dtype=np.float32) > 0
    out, cur, streak, st = [], None, 0, 0
    for i, v in enumerate(s.tolist()):
        if cur is None:
            cur = v
        elif v != cur:
            if streak == 0:
                st = i
            streak += 1
            if streak >= m:
                out.append(st)
                cur, streak = v, 0
        else:
            streak = 0
    return np.asarray(out, dtype=np.int64)


def histogram(d, fs: float):
    """Step 3: (H uint32 [Lmax + 1], long_runs)."""
    lmax, m = geometry(fs)
    L = np.diff(edges(d, m))
    inside = (L >= 1) & (L <= lmax)
    H = np.bincount(L[inside], minlength=lmax + 1).astype(np.uint32)
    return H, int((~inside).sum())


def score(H, long_runs: int, fs: float) -> dict:
    """Steps 4-5: the five fields of hbd_baud_estimate."""
    H = np.asarray(H, dtype=np.uint64)
    L = np.arange(H.size, dtype=np.int64)
    runs = int(H.sum())
    out = {"baud": 0.0, "nominal": 0.0, "confidence": 0.0, "runs": runs, "long_runs": int(long_runs)}
    cands = [b for b in CANDIDATES if fs / b >= 8]
    if not runs or not cands:
        return out
    sums = []
    for b in cands:
        sp = fs / b
        k = np.floor(L / sp + 0.5)
        ok = (k >= 1) & (k <= 6) & (np.abs(L - k * sp) <= 0.2 * sp)
        E = int(H[ok].sum())
        SK = int((H[ok] * k[ok].astype(np.uint64)).sum())
        SL = int((H[ok] * L[ok].astype(np.uint64)).sum())
        sums.append((b, E, SK, SL))
    emax = max(E for _, E, _, _ in sums)
    b, E, SK, SL = next(x for x in sums if 10 * x[1] >= 9 * emax)
    out.update(nominal=float(b), confidence=E / runs, baud=fs * float(SK) / float(SL) if SL else 0.0)
    return out


def estimate(d, fs: float) -> dict:
    H, long_runs = histogram(d, fs)
    return score(H, long_runs, fs)
