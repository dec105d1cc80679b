// RTTY tone-pair search on an averaged power spectrum (hbd_scan_detect, include/habdec_b200.h).  Host only, float64.
//
//   noise floor   lower median of the block of 1024 bins holding the bin
//   candidates    P[k] >= nf(k) 10^(min_snr/10) and the first maximum of P over [k-g, k+g], g = max(1, floor(min_shift / (2 fs/N)))
//   pairing       strongest unused candidate first (ties: lower bin); its partner is the strongest unused candidate
//                 min_shift <= |f_b - f_a| <= max_shift whose power is within max_tone_ratio of it; then every candidate in
//                 [f_lo - d, f_hi + d], d = f_hi - f_lo, is used up (the modulation sidelobes of the pair)
// tests/scan_ref.py restates these rules in numpy; the two must agree bin for bin.
#include "../../include/habdec_b200.h"

#include <algorithm>
#include <climits>
#include <cmath>
#include <vector>

extern "C" void hbd_scan_default_params(hbd_scan_params* p)
{
    if (!p) return;
    p->min_snr_db = 10.0;
    p->min_shift_hz = 150.0;
    p->max_shift_hz = 1200.0;
    p->max_tone_ratio_db = 15.0;   // the idle mark tone makes the two tones of a 50-baud payload differ by ~8 dB
}

extern "C" int hbd_scan_detect(const float* psd, size_t n, double fs, const hbd_scan_params* params, hbd_scan_signal* out, size_t cap)
{
    if (!psd || !n || n > size_t(INT_MAX) || !(fs > 0) || (cap && !out)) return HBD_ERR_ARG;
    hbd_scan_params p;
    hbd_scan_default_params(&p);
    if (params) p = *params;
    if (std::isnan(p.min_snr_db) || std::isnan(p.min_shift_hz) || std::isnan(p.max_shift_hz) || std::isnan(p.max_tone_ratio_db)) return HBD_ERR_ARG;
    const long long N = (long long)n;
    const double bw = fs / double(N);
    auto f = [&](long long i) { return double(i - N / 2) * bw; };
    auto P = [&](long long i) { return double(psd[i]); };

    std::vector<double> nf(static_cast<size_t>(N));
    {
        std::vector<float> blk;
        for (long long b = 0; b < N; b += 1024) {
            const long long e = std::min(N, b + 1024);
            blk.assign(psd + b, psd + e);
            std::sort(blk.begin(), blk.end());
            const double med = double(blk[(blk.size() - 1) / 2]);
            std::fill(nf.begin() + b, nf.begin() + e, med);
        }
    }
    const double thr = std::pow(10.0, p.min_snr_db / 10.0);
    const double gd = std::floor(p.min_shift_hz / (2.0 * fs / double(N)));
    const long long g = gd >= double(N) ? N : std::max(1LL, (long long)gd);
    std::vector<long long> cand;   // ascending bin
    for (long long k = 0; k < N; ++k) {
        const double pk = P(k);
        if (!(pk >= nf[size_t(k)] * thr)) continue;
        bool peak = true;
        for (long long j = std::max(0LL, k - g); j < k && peak; ++j) peak = pk > P(j);
        for (long long j = k + 1; j <= std::min(N - 1, k + g) && peak; ++j) peak = pk >= P(j);
        if (peak) cand.push_back(k);
    }

    const size_t C = cand.size();
    std::vector<size_t> order(C);
    for (size_t i = 0; i < C; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return P(cand[a]) > P(cand[b]) || (P(cand[a]) == P(cand[b]) && cand[a] < cand[b]); });
    std::vector<unsigned char> used(C, 0);
    const double ratio = std::pow(10.0, -p.max_tone_ratio_db / 10.0);
    // candidates whose bins lie in [lo, hi] (clamped), as indices into cand
    auto span = [&](double lo, double hi, size_t& i0, size_t& i1) {
        const long long blo = lo < -double(N) ? -N : (long long)std::floor(lo), bhi = hi > 2.0 * double(N) ? 2 * N : (long long)std::ceil(hi);
        i0 = size_t(std::lower_bound(cand.begin(), cand.end(), blo) - cand.begin());
        i1 = size_t(std::upper_bound(cand.begin(), cand.end(), bhi) - cand.begin());
    };
    struct Sig { double center, shift, snr; long long lo, hi; };
    std::vector<Sig> sig;
    for (size_t oi = 0; oi < C; ++oi) {
        const size_t ia = order[oi];
        if (used[ia]) continue;
        const long long a = cand[ia];
        const double pa = P(a), fa = f(a);
        // partner search over the bins the shift range can reach (two bins of slack for rounding; the test below is exact)
        const double reach = p.max_shift_hz / bw + 2.0;
        size_t i0, i1;
        span(double(a) - reach, double(a) + reach, i0, i1);
        long long best = -1;
        size_t ib = 0;
        for (size_t i = i0; i < i1; ++i) {
            if (i == ia || used[i]) continue;
            const long long b = cand[i];
            const double pb = P(b), d = std::fabs(f(b) - fa);
            if (!(p.min_shift_hz <= d && d <= p.max_shift_hz)) continue;
            if (!(std::min(pa, pb) >= std::max(pa, pb) * ratio)) continue;
            if (best < 0 || pb > P(best) || (pb == P(best) && b < best)) { best = b; ib = i; }
        }
        if (best < 0) continue;
        const double fb = f(best), pb = P(best);
        const double flo = std::min(fa, fb), fhi = std::max(fa, fb), d = fhi - flo;
        used[ia] = used[ib] = 1;
        const long long lo = std::min(a, best), hi = std::max(a, best);
        span(double(lo - (hi - lo)) - 2.0, double(hi + (hi - lo)) + 2.0, i0, i1);
        for (size_t i = i0; i < i1; ++i) {
            const double fc = f(cand[i]);
            if (flo - d <= fc && fc <= fhi + d) used[i] = 1;
        }
        const double snr = 10.0 * std::log10(std::min(pa / nf[size_t(a)], pb / nf[size_t(best)]));
        sig.push_back({(fa + fb) / 2.0, std::fabs(fb - fa), snr, lo, hi});
    }
    std::sort(sig.begin(), sig.end(), [](const Sig& x, const Sig& y) { return x.center < y.center || (x.center == y.center && x.lo < y.lo); });
    for (size_t i = 0; i < sig.size() && i < cap; ++i) {
        out[i].center_hz = sig[i].center; out[i].shift_hz = sig[i].shift; out[i].snr_db = sig[i].snr;
        out[i].bin_lo = int(sig[i].lo); out[i].bin_hi = int(sig[i].hi);
    }
    return int(std::min<size_t>(sig.size(), size_t(INT_MAX)));
}
