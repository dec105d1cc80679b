"""numpy float64 restatement of the wideband scanner (include/habdec_b200.h, hbd_scan_*): the averaged spectrum (Welch,
hop N/2, 4-term Blackman-Harris window) and the tone-pair detection on a given float32 PSD, written as plainly as the
rules read so that the library's C++ detection can be checked against it bin for bin."""
import math

import numpy as np

BH4 = (0.35874, 0.48829, 0.14128, 0.01168)      # habdec_windows.h:27-53, denominators N - 1
DEFAULTS = dict(min_snr_db=10.0, min_shift_hz=150.0, max_shift_hz=1200.0, max_tone_ratio_db=15.0)


def window(N):
    n = np.arange(N, dtype=np.float64)
    a0, a1, a2, a3 = BH4
    w = a0 - a1 * np.cos(2 * np.pi * n / (N - 1)) + a2 * np.cos(4 * np.pi * n / (N - 1)) - a3 * np.cos(6 * np.pi * n / (N - 1))
    return w.astype(np.float32).astype(np.float64)    # the library stores the window as float32


def welch(x, N):
    """(fft-shifted float64 PSD, segments): P[k] = sum_s |X_s[k]|^2 / (S sum w^2) over the complete segments [s N/2, s N/2 + N)."""
    x = np.asarray(x)
    w = window(N)
    hop = N // 2
    S = (len(x) - N) // hop + 1 if len(x) >= N else 0
    P = np.zeros(N)
    step = max(1, (1 << 22) // N)
    for s0 in range(0, S, step):
        idx = np.arange(s0, min(S, s0 + step))[:, None] * hop + np.arange(N)[None, :]
        X = np.fft.fft(w[None, :] * x[idx].astype(np.complex128), axis=1)
        P += (np.abs(X) ** 2).sum(axis=0)
    if S:
        P /= S * np.sum(w * w)
    return np.fft.fftshift(P), S


def detect(psd, fs, **params):
    """Signals [(center_hz, shift_hz, snr_db, bin_lo, bin_hi)] sorted by center_hz, by the rules of hbd_scan_detect."""
    p = dict(DEFAULTS, **params)
    P = [float(v) for v in np.asarray(psd, dtype=np.float32)]
    N = len(P)
    bw = fs / N

    def f(i):
        return float(i - N // 2) * bw

    nf = [0.0] * N
    for b in range(0, N, 1024):
        blk = sorted(P[b:b + 1024])
        med = blk[(len(blk) - 1) // 2]
        for k in range(b, min(N, b + 1024)):
            nf[k] = med
    thr = 10.0 ** (p["min_snr_db"] / 10.0)
    g = max(1, int(math.floor(p["min_shift_hz"] / (2.0 * fs / N))))
    cand = []
    for k in range(N):
        if not P[k] >= nf[k] * thr:
            continue
        if all(P[k] > P[j] for j in range(max(0, k - g), k)) and all(P[k] >= P[j] for j in range(k + 1, min(N, k + g + 1))):
            cand.append(k)
    order = sorted(cand, key=lambda k: (-P[k], k))
    ratio = 10.0 ** (-p["max_tone_ratio_db"] / 10.0)
    used = set()
    out = []
    for a in order:
        if a in used:
            continue
        best = None
        for b in cand:
            if b == a or b in used:
                continue
            d = abs(f(b) - f(a))
            if not (p["min_shift_hz"] <= d <= p["max_shift_hz"]):
                continue
            if not (min(P[a], P[b]) >= max(P[a], P[b]) * ratio):
                continue
            if best is None or P[b] > P[best] or (P[b] == P[best] and b < best):
                best = b
        if best is None:
            continue
        flo, fhi = min(f(a), f(best)), max(f(a), f(best))
        d = fhi - flo
        used.update((a, best))
        used.update(c for c in cand if flo - d <= f(c) <= fhi + d)
        snr = 10.0 * math.log10(min(P[a] / nf[a], P[best] / nf[best]))
        out.append(((f(a) + f(best)) / 2.0, abs(f(best) - f(a)), snr, min(a, best), max(a, best)))
    return sorted(out, key=lambda s: (s[0], s[3]))
