// Per-call AFC state machine (device functions shared by K2, which steps it on calls that complete no FFT frame, and K4)
#pragma once
#include "hbd_common.cuh"

namespace hbd {

// ---- Average<T> (Average.h:39-55) -------------------------------------------------------------------------------
__device__ __forceinline__ double avg_get_d(double sum, unsigned cnt) { return cnt ? __ddiv_rn(sum, double(cnt)) : sum; }
__device__ __forceinline__ double avg_add_d(double& sum, unsigned& cnt, unsigned cap, double val)
{
    const double g = avg_get_d(sum, cnt);
    const double diff = __dsub_rn(g, val);
    if (cnt == cap) sum = __dadd_rn(__dmul_rn(g, double(cap - 1)), val);
    else { ++cnt; sum = __dadd_rn(sum, val); }
    return diff;
}
__device__ __forceinline__ double avg_get_i(int sum, unsigned cnt) { return cnt ? __ddiv_rn(double(sum), double(cnt)) : double(sum); }
__device__ __forceinline__ double avg_add_i(int& sum, unsigned& cnt, unsigned cap, int val)
{
    const double g = avg_get_i(sum, cnt);
    const double diff = __dsub_rn(g, double(val));
    if (cnt == cap) sum = int(__dadd_rn(__dmul_rn(g, double(cap - 1)), double(val))); // truncating assignment
    else { ++cnt; sum += val; }
    return diff;
}

__device__ __forceinline__ void afc_step(ChanState& st, double fs_dec, int n_fft)
{
    if (!st.have_spectrum || !st.spec_ok) { st.afc_correction = 0; return; } // AFC.h:96-100
    st.afc_noise_floor = st.spec_nf;
    st.afc_noise_var = st.spec_nv;
    avg_add_d(st.nf_sum, st.nf_cnt, 100, st.spec_nf);
    avg_add_d(st.nv_sum, st.nv_cnt, 100, st.spec_nv);
    int p1 = st.spec_p1, p2 = st.spec_p2;
    const float thr = float(__dadd_rn(avg_get_d(st.nf_sum, st.nf_cnt), __dmul_rn(3.0, fabs(avg_get_d(st.nv_sum, st.nv_cnt)))));
    const bool d1 = st.spec_p1_val > thr, d2 = st.spec_p2_val > thr;
    bool stable_l = false, stable_r = false;
    if (d1 && d2) {
        if (p2 < p1) { const int t = p1; p1 = p2; p2 = t; }
        if (avg_add_i(st.pl_sum, st.pl_cnt, 4, p1) <= 2.0) stable_l = true;
        if (avg_add_i(st.pr_sum, st.pr_cnt, 4, p2) <= 2.0) stable_r = true;
    }
    const double la = avg_get_i(st.pl_sum, st.pl_cnt), ra = avg_get_i(st.pr_sum, st.pr_cnt);
    st.gui_left = 0;
    if (d1) st.gui_left = stable_l ? int(la) : int(-la);
    st.gui_right = 0;
    if (d2) st.gui_right = stable_r ? int(ra) : int(-ra);
    if (stable_l && stable_r) {
        const int pl = int(round(la)), pr = int(round(ra));
        const int dist = pr - pl;
        const double hz_per_bin = __ddiv_rn(fs_dec, double(n_fft));
        st.afc_shift_hz = __dmul_rn(hz_per_bin, double(dist));
        const double mid = double(pl + dist / 2);
        const double err = __dsub_rn(mid, double(n_fft) / 2);
        if (4 < fabs(err)) st.afc_correction = __dmul_rn(hz_per_bin, err);
    }
}


// the fields afc_step() modifies, copied from a staged ChanState back to the channel's state in HBM
__device__ __forceinline__ void afc_store(ChanState& dst, const ChanState& src)
{
    dst.afc_correction = src.afc_correction; dst.afc_noise_floor = src.afc_noise_floor; dst.afc_noise_var = src.afc_noise_var;
    dst.afc_shift_hz = src.afc_shift_hz;
    dst.nf_sum = src.nf_sum; dst.nf_cnt = src.nf_cnt; dst.nv_sum = src.nv_sum; dst.nv_cnt = src.nv_cnt;
    dst.pl_sum = src.pl_sum; dst.pl_cnt = src.pl_cnt; dst.pr_sum = src.pr_sum; dst.pr_cnt = src.pr_cnt;
    dst.gui_left = src.gui_left; dst.gui_right = src.gui_right;
}

// AFC::resetFrequencyCorrection (AFC.h:188-194): the peak averages move by `corr` Hz and restart, the correction is 0 again
__device__ __forceinline__ void afc_reset(ChanState& st, double corr, double fs_dec, int n_fft)
{
    // the reference divides fft_samples_.size() by its sampling rate: both are 0 before the first spectrum
    const double bins_per_hz = st.have_spectrum ? __ddiv_rn(double(n_fft), fs_dec) : __ddiv_rn(0.0, 0.0);
    const double l = __dsub_rn(avg_get_i(st.pl_sum, st.pl_cnt), __dmul_rn(corr, bins_per_hz));
    const double r = __dsub_rn(avg_get_i(st.pr_sum, st.pr_cnt), __dmul_rn(corr, bins_per_hz));
    st.pl_sum = int(fmax(0.0, l)); st.pl_cnt = 1;
    st.pr_sum = int(fmax(0.0, r)); st.pr_cnt = 1;
    st.afc_correction = 0;
}

} // namespace hbd
