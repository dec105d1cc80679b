"""hbd_reset_channels: listed channels start over like channel 0 of a new handle with the same settings, while the other
channels of the handle go on undisturbed, and batch / wideband calls after the reset are planned in O(1) of the channel
count again (frame levels)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from habdec_b200 import api, synth
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 65536
STAGES = (api.STAGE_DECIMATED, api.STAGE_FILTERED, api.STAGE_DEMOD, api.STAGE_LPTAPS, api.STAGE_PENDING, api.STAGE_BITS)


def rel_l2(a, b):
    a = np.asarray(a).astype(np.complex128 if np.iscomplexobj(a) else np.float64)
    b = np.asarray(b).astype(a.dtype)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def sentence(tag, c, k=0):
    body = "%s%02d,%d,12:00:%02d,%d" % (tag, c, k, c, 700 * c + k)   # > 20 characters (Decoder.h:591)
    return "$$" + body + "*" + synth.crc16_ccitt(body.encode()) + "\n"


# ---- 1. against the reference -----------------------------------------------------------------------------------------
FS = 2.5e6
OFF_A = [-600e3, -150e3, 420e3]     # payloads A, on the air from the start, one per channel
OFF_B = 830e3                       # payload B, launched at call K_RESET; channel RC is handed over to it
K_RESET, RC = 60, 1


def _reassign_capture():
    bits_a = [synth.uart_bits((sentence("PLA", c, 0) + sentence("PLA", c, 1)).encode(), 8, 2, 30, 40) for c in range(len(OFF_A))]
    bits_b = synth.uart_bits((sentence("PLB", 9, 0) + sentence("PLB", 9, 1)).encode(), 8, 2, 30, 40)
    n_b = int(len(bits_b) * FS / 300.0)
    n = (K_RESET * CHUNK + n_b) // CHUNK * CHUNK + CHUNK
    x = np.zeros(n, dtype=np.complex128)
    for c, (b, f) in enumerate(zip(bits_a, OFF_A)):
        x += synth.fsk_iq(b, FS, 300.0, 425.0, f, None, n_samples=n, phase0=0.3 * c)
    x[K_RESET * CHUNK:] += synth.fsk_iq(bits_b, FS, 300.0, 425.0, OFF_B, None, n_samples=n - K_RESET * CHUNK, phase0=1.1)
    rng = np.random.default_rng(11)
    sigma = 10.0 ** (8.0 / 20.0) / np.sqrt(2.0)
    x += sigma * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return x.astype(np.complex64)


def _reference(kind, x, f_hz):
    ref = (po.RefDecoder if kind == "ref" else po.PortDecoder)(po.make_config(baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=256))
    ph = 0.0
    for o in range(0, len(x), CHUNK):
        mixed, ph = po.premix(x[o:o + CHUNK], FS, f_hz, ph)
        ref.push_process(mixed, FS)
    return ref


@pytest.mark.parametrize("route", ["batch", "channel", "wideband_device", "cs16_device"])
def test_reset_and_retune_equals_new_reference_decoder(oracle_kind, route):
    import torch
    x = _reassign_capture()
    if route == "cs16_device":   # the decoder sees the dequantised values
        q = api.quantise(x, api.IQ_CS16, scale=1.0 / 16)
        x = api.dequantise(q, api.IQ_CS16)
        dev = torch.from_numpy(np.ascontiguousarray(q)).cuda()
    elif route == "wideband_device":
        dev = torch.from_numpy(x.view(np.float32)).cuda()
    torch.cuda.synchronize()
    n_ch, n = len(OFF_A), len(x)
    dec = api.BatchDecoder(n_ch, record=True, baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    for c, f in enumerate(OFF_A):
        dec.set_nco(f, c)
    post = {s: [] for s in (api.STAGE_DECIMATED, api.STAGE_DEMOD)}
    for k in range(n // CHUNK):
        o = k * CHUNK
        if k == K_RESET:
            before = dec.getRTTY(RC), dec.getLastSentence(RC)
            dec.reset_channels([RC])
            dec.set_nco(OFF_B, RC)
            pre_ref = _reference(oracle_kind, x[:o], OFF_A[RC])
            assert before == (pre_ref.rtty(), pre_ref.last_sentence())
            # decoded before the reset, polled after it: still queued, and nothing of the old text state is left
            assert dec.poll_chars(RC) == pre_ref.chars() and len(pre_ref.chars()) > 30
            assert dec.poll_sentences(RC) == pre_ref.sentences() and len(pre_ref.sentences()) >= 1
            assert dec.getRTTY(RC) == b"" and dec.getLastSentence(RC) == b""
            assert dec.getPowerSpectrum(RC).size == 0 and dec.getPeaks(RC) == (0, 0)
        if route == "batch":
            dec.pushSamplesBatch(np.ascontiguousarray(np.broadcast_to(x[o:o + CHUNK], (n_ch, CHUNK))), FS)
        elif route == "channel":
            for c in range(n_ch):
                dec.pushSamples(c, x[o:o + CHUNK], FS)
        elif route == "wideband_device":
            dec.pushWidebandDevice(dev.data_ptr() + o * 8, CHUNK, FS)
        else:
            dec.pushIQWidebandDevice(dev.data_ptr() + o * 4, api.IQ_CS16, CHUNK, FS)
        dec.process()
        if k >= K_RESET:
            for s in post:
                post[s].append(dec.debug_stage(RC, s).copy())
    ref_b = _reference(oracle_kind, x[K_RESET * CHUNK:], OFF_B)
    for s, which in ((api.STAGE_DECIMATED, po.STAGE_DECIMATED), (api.STAGE_DEMOD, po.STAGE_DEMOD)):
        want, at = ref_b.stage(which), 0
        for blk in post[s]:
            if blk.size:
                assert rel_l2(blk, want[at:at + blk.size]) <= 1e-5, "stage %d, call at %d" % (s, at)
            at += blk.size
        assert at == want.size
    assert dec.poll_chars(RC) == ref_b.chars()
    assert dec.poll_sentences(RC) == ref_b.sentences() == [sentence("PLB", 9, k).strip()[2:].encode() for k in range(2)]
    assert dec.getRTTY(RC) == ref_b.rtty() and dec.getLastSentence(RC) == ref_b.last_sentence()
    assert (n // CHUNK - K_RESET) * CHUNK // 256 >= 2 * 4096   # at least two spectrum frames since the reset
    a = ref_b.afc()
    assert dec.getPeaks(RC) == (a.peak_left, a.peak_right)
    for c in range(n_ch):
        if c == RC:
            continue
        ref = _reference(oracle_kind, x, OFF_A[c])
        assert dec.poll_chars(c) == ref.chars() and dec.poll_sentences(c) == ref.sentences() and len(ref.sentences()) == 2
        assert dec.getRTTY(c) == ref.rtty()


# ---- 2. a reset channel equals the same channel of a new handle, bit for bit ------------------------------------------
def _make(n_ch, factor, trans):
    d = api.BatchDecoder(n_ch, record=True, baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=factor, lowpass_trans=trans)
    d.set_ssdv(True); d.set_demod_accumulate(True); d.set_raw_chars(True)
    return d


def _snapshot(d, c):
    info, power = d.getSpectrumInfo(c)
    return ([d.debug_stage(c, s).tobytes() for s in STAGES], d.getFFT(c).tobytes(), d.getPowerSpectrum(c).tobytes(), bytes(info), power.tobytes(),
            d.spectrum_frame(c, 1.0, 512, 2), d.demod_frame(c, 300, 4),
            np.array(d.getNoiseFloor(c) + (d.getShift(c), d.getFrequencyCorrection(c)), dtype=np.float64).tobytes())


def _results(d, c):
    pk = d.poll_ssdv_packets(c)
    return (d.poll_chars(c), d.poll_sentences(c), d.poll_raw_chars(c), d.getRTTY(c), d.getLastSentence(c), pk,
            [d.get_ssdv_image(c, p[0], p[1]) for p in pk])


# Factor 256 (PHASE_256 of test_gpu_call_paths): before the reset a redesign and a push that leaves a carry remainder; after
# it buffer growth, a gated call, a call with no decimation block and redesigns.  Cascade: setupDecimationStagesBW(600).
PRE_256 = [(65536, None)] * 3 + [(65536, 0.05), (100000, None), (10000, None), (65536, None)]
POST_256 = [(65536, None), (100, None), (100000, None), (10000, None), (131072, 0.0125), (65536, 0.025)] + [(65536, None)] * 40
PRE_CASCADE = [(65536, None), (262144, None), (65536, None)]
POST_CASCADE = [(262144, None), (524288, 0.05), (65536, None), (1000000, None)] + [(65536, None)] * 10


@pytest.mark.parametrize("sched,reset", [("f256", (1, 3)), ("cascade", (1, 3)), ("f256", (0, 1, 2, 3))])
def test_reset_equals_new_handle(sched, reset):
    fs, n_ch = 2.048e6, 4
    pre, post = (PRE_256, POST_256) if sched == "f256" else (PRE_CASCADE, POST_CASCADE)
    total = sum(n for n, _ in pre + post)
    iq = np.stack([synth.channel_iq(40 + c, 3, fs, 300.0, snr_db=-12.0, n_samples=total)[0] for c in range(n_ch)])
    trans = 0.025
    a, c_ = _make(n_ch, 256, trans), _make(n_ch, 256, trans)   # a: reset at the boundary; c_: never reset
    b, o = None, 0

    def step(decs, n, t):
        nonlocal o, trans
        if t is not None:
            trans = t
            for d in decs:
                d.lowpass_trans(t, -1)
        blk = np.ascontiguousarray(iq[:, o:o + n])
        o += n
        for d in decs:
            d.pushSamplesBatch(blk, fs)
            if sched == "cascade" and d.getDecimationFactor() == 256:
                assert d.setupDecimationStagesBW(600.0) == 4096
            d.process()

    for n, t in pre:
        step((a, c_), n, t)
    for d in (a, c_):   # output decoded before the reset is not compared (channel a differs from b there)
        for ch in range(n_ch):
            _results(d, ch)
    a.reset_channels(list(reset))
    assert a.getRTTY(reset[0]) == b"" and a.getPowerSpectrum(reset[0]).size == 0
    b = _make(n_ch, 256, trans)
    a.set_kernel_timing(1); b.set_kernel_timing(1)
    for i, (n, t) in enumerate(post):
        step((a, b, c_), n, t)
        for ch in range(n_ch):
            want = b if ch in reset else c_
            assert _snapshot(a, ch) == _snapshot(want, ch), "call %d after the reset: channel %d" % (i, ch)
    for ch in range(n_ch):
        got, want = _results(a, ch), _results(b if ch in reset else c_, ch)
        assert got == want, "channel %d" % ch
    if sched == "f256":   # (the cascade decimates to 500 Hz: nothing to decode at 300 baud, only the state to compare)
        assert all(len(a.getRTTY(ch)) > 10 for ch in range(n_ch))
    if len(reset) == n_ch:   # every channel reset: back to one frame level, planned once per call like the new handle
        assert a.kernel_timing(6)[1] == b.kernel_timing(6)[1] == len(post)


# ---- 3. uniform planning survives resets --------------------------------------------------------------------------------
def test_uniform_planning_after_resets():
    fs, n_ch, n_calls = 2.048e6, 64, 60
    resets = {3: [5, 17], 9: [2], 14: [40, 41, 63], 22: [17], 29: [0, 33]}   # 5 calls, 5 different frame phases
    rng = np.random.default_rng(3)
    base = np.stack([synth.channel_iq(c % 8, 1, fs, 300.0, snr_db=-10.0, n_samples=n_calls * CHUNK)[0] for c in range(8)])
    uni, per = (api.BatchDecoder(n_ch, record=True, dec_factor=256) for _ in range(2))
    for d in (uni, per):
        d.set_kernel_timing(1)
    fill = np.zeros(n_ch, dtype=np.int64)
    last = max(resets)
    deltas = {uni: [], per: []}
    for k in range(n_calls):
        if k in resets:
            for d in (uni, per):
                d.reset_channels(resets[k])
            fill[resets[k]] = 0
        blk = np.ascontiguousarray(base[np.arange(n_ch) % 8, k * CHUNK:(k + 1) * CHUNK])
        blk *= (1.0 + 0.01 * rng.standard_normal((n_ch, 1))).astype(np.float32)
        uni.pushSamplesBatch(blk, fs)
        for c in range(n_ch):
            per.pushSamples(c, blk[c], fs)
        for d in (uni, per):
            t0 = d.kernel_timing(6)[1]
            l0 = d.kernel_launches()
            d.process()
            deltas[d].append((d.kernel_launches() - l0, d.kernel_timing(6)[1] - t0))
        fill += 256
        k4 = bool((fill >= 4096).any())
        fill[fill >= 4096] = 0
        deltas[uni][-1] += (k4,)
        if k >= last + 1:   # from the second call after the last reset on (the first one plans every channel on its own)
            assert deltas[uni][-1][1] <= 6, "call %d: %d counters stepped" % (k, deltas[uni][-1][1])
        assert deltas[per][-1][1] == n_ch
        for c in range(0, n_ch, 7):
            assert uni.debug_stage(c, api.STAGE_DEMOD).tobytes() == per.debug_stage(c, api.STAGE_DEMOD).tobytes()
    steady = [x for k, x in enumerate(deltas[uni]) if k >= last + 1]
    base_launches = min(x[0] for x in steady)
    assert [x[0] - base_launches for x in steady] == [int(x[2]) for x in steady]   # K4 exactly on the frame-completing calls
    assert any(x[2] for x in steady) and not all(x[2] for x in steady)
    assert [x[0] for x in deltas[uni]] == [x[0] for x in deltas[per]]
    for c in range(n_ch):
        assert uni.poll_chars(c) == per.poll_chars(c) and uni.poll_sentences(c) == per.poll_sentences(c)
        assert uni.getPeaks(c) == per.getPeaks(c)
        for s in STAGES:
            assert uni.debug_stage(c, s).tobytes() == per.debug_stage(c, s).tobytes()


# ---- 4. pipelined use ---------------------------------------------------------------------------------------------------
def test_pipelined_resets_equal_synchronous():
    fs, n_ch, n_calls = 2.048e6, 6, 70
    iq = np.stack([synth.channel_iq(20 + c, 2, fs, 300.0, snr_db=-10.0, n_samples=n_calls * CHUNK)[0] for c in range(n_ch)])
    resets = {25: [1, 4], 41: [2], 55: [1]}
    sync, pipe = api.BatchDecoder(n_ch), api.BatchDecoder(n_ch)
    cbs = {sync: [b""] * n_ch, pipe: [b""] * n_ch}
    sents = {sync: [[] for _ in range(n_ch)], pipe: [[] for _ in range(n_ch)]}
    for d in (sync, pipe):
        def on_chars(ch, s, d=d): cbs[d][ch] += s
        def on_sent(ch, cs, data, crc, d=d): sents[d][ch].append((cs, data, crc))
        d.set_chars_callback(on_chars); d.set_sentence_callback(on_sent)
    for k in range(n_calls):
        if k in resets:
            sync.reset_channels(resets[k])
            pipe.reset_channels(resets[k])
            # the drain inside the reset fired the callbacks of everything decoded so far before returning
            assert cbs[pipe] == cbs[sync] and sents[pipe] == sents[sync]
        blk = np.ascontiguousarray(iq[:, k * CHUNK:(k + 1) * CHUNK])
        sync.pushSamplesBatch(blk, fs); sync.process()
        pipe.pushSamplesBatch(blk, fs); pipe.process_async(); pipe.collect_ready(3)
    pipe.collect()
    assert cbs[pipe] == cbs[sync] and sents[pipe] == sents[sync]
    for c in range(n_ch):
        assert pipe.poll_chars(c) == sync.poll_chars(c) == cbs[sync][c]
        assert pipe.poll_sentences(c) == sync.poll_sentences(c)
        assert pipe.getRTTY(c) == sync.getRTTY(c)
    assert sum(len(s) for s in sents[sync]) >= 2


# ---- 5. errors ------------------------------------------------------------------------------------------------------------
def test_errors_change_nothing():
    import torch
    fs, n_ch = 2.048e6, 3
    iq = np.stack([synth.channel_iq(60 + c, 1, fs, 300.0, snr_db=-10.0, n_samples=30 * CHUNK)[0] for c in range(n_ch)])
    lib = api.load()
    x, y = api.BatchDecoder(n_ch, record=True), api.BatchDecoder(n_ch, record=True)
    h = x._h

    def rc(chs):
        arr = (C.c_int * max(len(chs), 1))(*chs)
        return lib.hbd_reset_channels(h, arr, len(chs))

    assert rc([]) == api.HBD_OK and lib.hbd_reset_channels(h, None, 0) == api.HBD_OK   # no-op
    assert lib.hbd_reset_channels(h, None, 1) == api.HBD_ERR_ARG
    assert lib.hbd_reset_channels(None, None, 0) == api.HBD_ERR_ARG
    dev = torch.from_numpy(np.ascontiguousarray(iq[:, 10 * CHUNK:11 * CHUNK]).view(np.float32)).cuda()
    torch.cuda.synchronize()
    launches = x.kernel_launches()
    for k in range(30):
        blk = np.ascontiguousarray(iq[:, k * CHUNK:(k + 1) * CHUNK])
        for chs in ([-1], [n_ch], [0, 2, 0], [1, 1]):
            assert rc(chs) == api.HBD_ERR_ARG
        if k == 10:   # a pending device input
            x.pushSamplesDevice(dev.data_ptr(), CHUNK, CHUNK, fs)
            assert rc([0]) == api.HBD_ERR_STATE
        elif k % 3 == 0:   # staged host samples, in every channel or in one
            x.pushSamplesBatch(blk, fs)
            assert rc([1]) == api.HBD_ERR_STATE
        else:
            for c in range(n_ch):
                x.pushSamples(c, blk[c], fs)
                assert rc([c]) == api.HBD_ERR_STATE
        assert x.kernel_launches() == launches
        y.pushSamplesBatch(blk, fs)
        x.process(); y.process()
        launches = x.kernel_launches()
        for c in range(n_ch):
            for s in STAGES:
                assert x.debug_stage(c, s).tobytes() == y.debug_stage(c, s).tobytes(), (k, c, s)
    for c in range(n_ch):
        assert x.poll_chars(c) == y.poll_chars(c) and x.getRTTY(c) == y.getRTTY(c) and len(y.getRTTY(c)) > 10
    # before the first push
    z = api.BatchDecoder(2)
    z.reset_channels([0, 1])
    z.pushSamplesBatch(np.ascontiguousarray(iq[:2, :CHUNK]), fs); z.process()


# ---- 6. C++ facade ------------------------------------------------------------------------------------------------------
def test_cpp_facade_reset_channels(tmp_path):
    fs, n_ch, n_calls, k_reset = 2.048e6, 2, 40, 17
    iq = np.stack([synth.channel_iq(70 + c, 2, fs, 300.0, snr_db=-10.0, n_samples=n_calls * CHUNK)[0] for c in range(n_ch)])
    path = str(tmp_path / "batch.cf32")
    np.ascontiguousarray(iq).tofile(path)
    exe = str(tmp_path / "reset_channels")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    lib_dir = os.path.join(ROOT, "habdec_b200")
    subprocess.run([cxx, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "reset_channels.cpp"),
                    "-L", lib_dir, "-lhabdec_b200", "-Wl,-rpath," + lib_dir, "-lpthread", "-o", exe], check=True)
    out = subprocess.run([exe, path, str(n_ch), str(n_calls * CHUNK), repr(fs), str(k_reset)], check=True, capture_output=True).stdout
    d = api.BatchDecoder(n_ch)
    want = b""
    for k in range(n_calls):
        if k == k_reset:
            want += b"PRE %s\n" % d.poll_chars(1).hex().encode()
            d.reset_channels([1])
        d.pushSamplesBatch(np.ascontiguousarray(iq[:, k * CHUNK:(k + 1) * CHUNK]), fs)
        d.process()
    for c in range(n_ch):
        want += b"CH%d %s %s\n" % (c, d.poll_chars(c).hex().encode(), d.getRTTY(c).hex().encode())
    assert out == want
    assert b"PRE \n" not in out
