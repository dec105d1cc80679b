"""Reading decoder state back to the host: the per-channel getters, hbd_get_spectrum_info, hbd_get_stats_batch and the
AFC scalars of hbd_pack_results report the same values, reading launches no kernel, and invalid handles or channels get
each entry point's fallback."""
import ctypes as C

import numpy as np
import pytest

from habdec_b200 import api, synth

pytestmark = pytest.mark.gpu

FS, CHUNK, N_CH, CALLS = 2.048e6, 65536, 8, 40
SIG_HZ = [-610e3, -95e3, 240e3, 730e3]
# four channels a few hundred Hz off a payload (so the AFC has a correction to report) and four on noise
NCO_HZ = [SIG_HZ[0] + 180.0, SIG_HZ[1] - 260.0, SIG_HZ[2] + 90.0, SIG_HZ[3] - 140.0, -850e3, -400e3, 120e3, 900e3]


@pytest.fixture(scope="module")
def capture():
    n = (CALLS + 1) * CHUNK
    x = np.zeros(n, dtype=np.complex64)
    for k, f in enumerate(SIG_HZ):
        bits = synth.uart_bits((synth.make_sentence(k, 0) * 3).encode())
        x += synth.fsk_iq(bits, FS, 300.0, 425.0, f, None, n_samples=n, phase0=0.4 * k)
    rng = np.random.default_rng(5)
    x.real += (0.3 * rng.standard_normal(n)).astype(np.float32)
    x.imag += (0.3 * rng.standard_normal(n)).astype(np.float32)
    return x


def decoded(capture, calls=CALLS):
    dec = api.BatchDecoder(N_CH, dec_factor=256)
    for c, f in enumerate(NCO_HZ):
        dec.set_nco(f, c)
    for k in range(calls):
        dec.pushWideband(capture[k * CHUNK:(k + 1) * CHUNK], FS)
        dec.process()
    return dec


@pytest.fixture(scope="module")
def dec(capture):
    return decoded(capture)


def test_getters_agree_and_launch_nothing(dec):
    launches = dec.kernel_launches()
    stats = dec.stats_all()
    assert stats.shape == (N_CH, 6)
    for c in range(N_CH):
        pl, pr = dec.getPeaks(c)
        nf, nv = dec.getNoiseFloor(c)
        corr, shift = dec.getFrequencyCorrection(c), dec.getShift(c)
        assert stats[c].tolist() == [corr, shift, nf, nv, pl, pr], "channel %d" % c

        pw = dec.getPowerSpectrum(c)
        assert pw.size == dec.getBinsCount() and dec.getFFT(c).size == dec.getBinsCount()
        info, power = dec.getSpectrumInfo(c)
        assert power.tobytes() == pw.tobytes()
        assert (info.min_, info.max_) == (pw.min(), pw.max())
        assert (info.peak_left_, info.peak_left_valid_) == (abs(pl), int(pl > 0))
        assert (info.peak_right_, info.peak_right_valid_) == (abs(pr), int(pr > 0))
        assert (info.noise_floor_, info.noise_variance_) == (nf, nv)
        assert info.sampling_rate_ == dec.getDecimatedSamplingRate()
        assert info.shift_ == shift
        assert dec.getDemodulated(c).size > 0
    assert dec.kernel_launches() == launches
    # the comparison means something: payload channels have locked on with an offset to correct
    assert (stats[:4, 4] > 0).all() and (stats[:4, 5] > 0).all() and (stats[:4, 0] != 0).all(), stats


def _records(recs):
    return [api.ResultRecord.from_buffer_copy(recs[c].tobytes()) for c in range(recs.shape[0])]


def _assert_scalars(recs, stats):
    want = stats.astype(np.float32)
    for c, r in enumerate(_records(recs)):
        assert [r.frequency_correction, r.shift, r.noise_floor, r.noise_variance] == want[c, :4].tolist(), "channel %d" % c
        assert (r.peak_left, r.peak_right) == (int(stats[c, 4]), int(stats[c, 5])), "channel %d" % c


def test_pack_results_live_then_snapshot(capture):
    d = decoded(capture)
    _assert_scalars(d.pack_results(), d.stats_all())   # never packed: no snapshot, the live state is read
    d.pushWideband(capture[CALLS * CHUNK:], FS)
    d.process()
    d.collect()
    _assert_scalars(d.pack_results(), d.stats_all())   # the snapshot of the drained call


def test_no_spectrum_yet(capture):
    d = decoded(capture, calls=1)   # 256 decimated samples: no FFT frame yet
    assert d.getFFT(0).size == 0 and d.getPowerSpectrum(0).size == 0
    info = api.SpectrumInfo(min_=1.0, max_=2.0, noise_floor_=3.0, shift_=4.0, peak_left_=5, peak_right_valid_=1)
    power = np.ones(d.getBinsCount(), dtype=np.float32)
    assert d._lib.hbd_get_spectrum_info(d._h, 0, C.byref(info), power.ctypes.data, power.size) == 0
    assert bytes(info) == bytes(api.SpectrumInfo())
    assert (power == 1).all()


def test_invalid_handle_and_channel(dec):
    lib, h, ERR = dec._lib, dec._h, api.HBD_ERR_ARG
    launches = dec.kernel_launches()
    i, d, info = C.c_int(7), C.c_double(7.0), api.SpectrumInfo()
    queries = {   # entry point -> what it returns for an invalid handle or channel
        "hbd_get_fft": (lambda h, c: lib.hbd_get_fft(h, c, None, 0), 0),
        "hbd_get_power_spectrum": (lambda h, c: lib.hbd_get_power_spectrum(h, c, None, 0), 0),
        "hbd_get_demodulated": (lambda h, c: lib.hbd_get_demodulated(h, c, None, 0), 0),
        "hbd_get_peaks": (lambda h, c: lib.hbd_get_peaks(h, c, C.byref(i), C.byref(i)), ERR),
        "hbd_get_noise_floor": (lambda h, c: lib.hbd_get_noise_floor(h, c, C.byref(d), C.byref(d)), ERR),
        "hbd_get_shift": (lambda h, c: lib.hbd_get_shift(h, c), 0.0),
        "hbd_get_frequency_correction": (lambda h, c: lib.hbd_get_frequency_correction(h, c), 0.0),
        "hbd_reset_frequency_correction": (lambda h, c: lib.hbd_reset_frequency_correction(h, c, 10.0), ERR),
        "hbd_get_spectrum_info": (lambda h, c: lib.hbd_get_spectrum_info(h, c, C.byref(info), None, 0), 0),
        "hbd_debug_stage": (lambda h, c: lib.hbd_debug_stage(h, c, api.STAGE_DEMOD, None, 0), 0),
        "hbd_get_spectrum_frame": (lambda h, c: lib.hbd_get_spectrum_frame(h, c, 1.0, 256, 1, None, 0), 0),
        "hbd_get_demod_frame": (lambda h, c: lib.hbd_get_demod_frame(h, c, 256, 1, None, 0), 0),
    }
    for name, (call, fallback) in queries.items():
        for hh, c in ((None, 0), (h, -1), (h, N_CH)):
            assert call(hh, c) == fallback, "%s(%s, %d)" % (name, "h" if hh else "NULL", c)
    assert (i.value, d.value) == (7, 7.0)
    assert lib.hbd_get_stats_batch(None, None, 0) == 0 and lib.hbd_get_stats_batch(h, None, 0) == 6 * N_CH
    assert lib.hbd_pack_results(None, 0, None, 0) == 0 and lib.hbd_pack_results(h, 0, None, 0) == N_CH
    assert dec.kernel_launches() == launches
