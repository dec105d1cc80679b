"""A process call steps the host counters in one of two ways.  After batch pushes (uniform mode) channel 0's counters stand
for every channel and the side effects of the step (history zeroing, low-pass tap uploads) are applied to all rows at once;
after per-channel pushes every channel is stepped and its side effects are applied to its own row.  Fed the same samples
in the same chunk sizes, both ways must give bit for bit the same results."""
import numpy as np
import pytest

from habdec_b200 import api, synth

pytestmark = pytest.mark.gpu

STAGES = (api.STAGE_DECIMATED, api.STAGE_FILTERED, api.STAGE_DEMOD, api.STAGE_LPTAPS, api.STAGE_PENDING, api.STAGE_BITS)

# (chunk size, lowpass_trans set for all channels before the call, or None).  Factor 256: the first call and the larger
# calls grow the work buffers (carry, stage-2 and low-pass history zeroed; 100 000 leaves a remainder in the carry, so the
# carry history sits at another offset), 100 samples make no decimation block, 10 000 leave the low-pass gated, and the
# low-pass is redesigned shorter, then longer than its work buffer (zeroed), then shorter again.
PHASE_256 = ([(65536, None)] * 4 + [(65536, 0.05), (100, None), (10000, None), (65536, 0.0125), (100000, None),
                                    (131072, None), (200000, None), (65536, 0.025)] + [(65536, None)] * 40)
# after setupDecimationStagesBW(600): factor 4096 = 64 (K1), 4, 8 (middle stages), 2 (tail kernel); the growing calls
# zero the histories of both middle stages
PHASE_CASCADE = [(65536, None), (262144, None), (524288, None), (65536, None), (262144, 0.05), (1000000, None), (65536, None)]


def stage_arrays(dec, n_ch):
    return [[dec.debug_stage(c, s).tobytes() for s in STAGES] for c in range(n_ch)]


def test_per_channel_calls_equal_uniform_calls():
    fs, baud, n_ch = 2.048e6, 300.0, 4
    total = sum(n for n, _ in PHASE_256 + PHASE_CASCADE)
    iq = np.stack([synth.channel_iq(80 + c, 2, fs, baud, snr_db=-12.0, n_samples=total)[0] for c in range(n_ch)])
    cfg = dict(baud=baud, rtty_bits=8, rtty_stops=2.0, dec_factor=256, record=True)
    uni, per = api.BatchDecoder(n_ch, **cfg), api.BatchDecoder(n_ch, **cfg)   # batch pushes / pushSamples(ch, ...)
    launches0 = (uni.kernel_launches(), per.kernel_launches())
    o = 0
    for phase, schedule in enumerate((PHASE_256, PHASE_CASCADE)):
        if phase == 1:
            assert uni.setupDecimationStagesBW(600.0) == per.setupDecimationStagesBW(600.0) == 4096
        for i, (n, trans) in enumerate(schedule):
            if trans is not None:
                uni.lowpass_trans(trans, -1); per.lowpass_trans(trans, -1)
            blk = np.ascontiguousarray(iq[:, o:o + n])
            o += n
            uni.pushSamplesBatch(blk, fs)
            for c in range(n_ch):
                per.pushSamples(c, blk[c], fs)
            uni.process(); per.process()
            a, b = stage_arrays(uni, n_ch), stage_arrays(per, n_ch)
            for c in range(n_ch):
                for s, x, y in zip(STAGES, a[c], b[c]):
                    assert x == y, "phase %d call %d (%d samples): channel %d, stage %d differs" % (phase, i, n, c, s)
    assert o == total
    chars = [uni.poll_chars(c) for c in range(n_ch)]
    assert chars == [per.poll_chars(c) for c in range(n_ch)]
    assert [uni.poll_sentences(c) for c in range(n_ch)] == [per.poll_sentences(c) for c in range(n_ch)]
    assert uni.kernel_launches() - launches0[0] == per.kernel_launches() - launches0[1]
    assert all(len(x) >= 10 for x in chars), "the schedule decodes too little to compare"
