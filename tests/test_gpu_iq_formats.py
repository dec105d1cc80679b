"""Integer IQ input (hbd_push_iq*, include/habdec_b200.h): an integer push is bit for bit the cf32 push of its dequantised
values.  Two handles in one process, one fed cf32 of api.dequantise(q), one fed q itself through the matching integer entry
point; every stage array, spectrum, AFC scalar and character must agree bitwise.  Plus the reference on integer rings at
full width (the native K1 path) and the C++ example on an rtl_sdr-style .cu8 file."""
import os
import subprocess

import numpy as np
import pytest

from habdec_b200 import api, synth
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FORMATS = [api.IQ_CS16, api.IQ_CS8, api.IQ_CU8]
FMT_ID = {api.IQ_CS16: "cs16", api.IQ_CS8: "cs8", api.IQ_CU8: "cu8"}
CHUNKS = [65536, 40001, 1, 0, 262144]          # odd, not a multiple of 4 or 8, single sample, empty push
SCALE = 1.0 / 32.0                              # synth signals at these SNRs stay well inside full scale
N_CH = 3
NCO_HZ = [20e3, 0.0, -35e3]


def _signals(fs, wide):
    if wide:
        row, _ = synth.channel_iq(2, 1, fs, 300.0, f_off=20e3, snr_db=-10.0)
        return row[None, :]
    sig = [synth.channel_iq(c, 1, fs, 300.0, snr_db=-10.0)[0] for c in range(N_CH)]
    n = min(len(s) for s in sig)
    return np.stack([s[:n] for s in sig])


def _plan_setup(plan):
    """(fs, factor for the constructor, cascade limit applied after a first one-sample call or None)"""
    return {"f256": (2.048e6, 256, None), "f32": (256e3, 32, None), "bw": (2.048e6, 1, 3000.0)}[plan]


def _chunks(n, first=None):
    out, o, i = [], 0, 0
    if first:
        out.append((0, first)); o = first
    while o < n:
        k = min(CHUNKS[i % len(CHUNKS)], n - o)
        out.append((o, k)); o += k; i += 1
    return out


class _Dev:
    """Aligned device staging for device pushes: a chunk is copied to the start of 16-byte aligned rows."""
    def __init__(self, torch, rows, cap, dtype, per_sample):
        self.t = torch.zeros((rows, (cap + 8) * per_sample), dtype=dtype, device="cuda")
        self.per = per_sample

    def put(self, torch, arr2d):
        k = arr2d.shape[1]
        if k:
            self.t[:, :k].copy_(torch.from_numpy(np.ascontiguousarray(arr2d)))
        torch.cuda.synchronize()
        return self.t.data_ptr(), self.t.shape[1] // self.per


def _compare(a, b, n_ch, where):
    for c in range(n_ch):
        for st in (api.STAGE_DECIMATED, api.STAGE_FILTERED, api.STAGE_DEMOD):
            x, y = a.debug_stage(c, st), b.debug_stage(c, st)
            assert x.shape == y.shape and np.array_equal(np.ascontiguousarray(x).view(np.uint32), np.ascontiguousarray(y).view(np.uint32)), \
                "%s ch %d stage %d" % (where, c, st)
        assert np.array_equal(a.getPowerSpectrum(c).view(np.uint32), b.getPowerSpectrum(c).view(np.uint32)), "%s ch %d spectrum" % (where, c)
        assert a.getPeaks(c) == b.getPeaks(c), where
        assert a.getFrequencyCorrection(c) == b.getFrequencyCorrection(c), where


def _finish(a, b, n_ch):
    for c in range(n_ch):
        assert a.poll_chars(c) == b.poll_chars(c)
        assert a.poll_sentences(c) == b.poll_sentences(c)
        assert a.poll_raw_chars(c) == b.poll_raw_chars(c)


def _pair(plan, n_ch, nco=None):
    fs, factor, _ = _plan_setup(plan)
    decs = [api.BatchDecoder(n_ch, baud=300.0, dec_factor=factor, record=True) for _ in range(2)]
    if nco:
        for d in decs:
            for c in range(n_ch):
                d.set_nco(nco[c], c)
    return decs


@pytest.mark.parametrize("plan", ["f256", "f32", "bw"])
@pytest.mark.parametrize("entry", ["host", "batch", "device", "wideband", "wideband_device"])
@pytest.mark.parametrize("fmt", FORMATS, ids=lambda f: FMT_ID[f])
def test_integer_push_is_the_cf32_push_of_its_values(fmt, entry, plan):
    import torch
    fs, _, bw = _plan_setup(plan)
    wide = entry.startswith("wideband")
    x = _signals(fs, wide)
    q = api.quantise(x, fmt, SCALE)                      # [rows, 2n]
    deq = api.dequantise(q, fmt)                         # [rows, n] complex64
    n = deq.shape[1]
    a, b = _pair(plan, N_CH, NCO_HZ if wide else None)
    dev_a = _Dev(torch, deq.shape[0], max(CHUNKS), torch.float32, 2) if entry.endswith("device") else None
    dev_b = _Dev(torch, deq.shape[0], max(CHUNKS), {api.IQ_CS16: torch.int16, api.IQ_CS8: torch.int8, api.IQ_CU8: torch.uint8}[fmt], 2) \
        if entry.endswith("device") else None
    for i, (o, k) in enumerate(_chunks(n, 1 if bw else None)):
        xa, xb = deq[:, o:o + k], q[:, 2 * o:2 * (o + k)]
        if entry == "host":
            for c in range(N_CH):
                a.pushSamples(c, xa[c], fs); b.pushIQ(c, xb[c], fmt, fs)
        elif entry == "batch":
            a.pushSamplesBatch(xa, fs); b.pushIQBatch(xb, fmt, fs)
        elif entry == "device":
            pa, pitch_a = dev_a.put(torch, xa.view(np.float32))
            pb, pitch_b = dev_b.put(torch, xb)
            a.pushSamplesDevice(pa, k, pitch_a, fs); b.pushIQDevice(pb, fmt, k, pitch_b, fs)
        elif entry == "wideband":
            a.pushWideband(xa[0], fs); b.pushIQWideband(xb[0], fmt, fs)
        else:
            pa, _ = dev_a.put(torch, xa.view(np.float32))
            pb, _ = dev_b.put(torch, xb)
            a.pushWidebandDevice(pa, k, fs); b.pushIQWidebandDevice(pb, fmt, k, fs)
        a.process(); b.process()
        if bw and i == 0:
            assert a.setupDecimationStagesBW(bw) == b.setupDecimationStagesBW(bw) == 1024
        _compare(a, b, N_CH, "call %d (chunk %d)" % (i, k))
    _finish(a, b, N_CH)


def test_native_k1_takes_no_widen_launch():
    """A CS16 device push at factor 256 is read by K1 itself: per call it launches exactly the kernels of the cf32 device push."""
    import torch
    fs = 2.048e6
    x = _signals(fs, False)[:, :8 * 65536]
    q = api.quantise(x, api.IQ_CS16, SCALE)
    deq = api.dequantise(q, api.IQ_CS16)
    a, b = _pair("f256", N_CH)
    ta = torch.from_numpy(deq.view(np.float32)).cuda()
    tb = torch.from_numpy(q).cuda()
    torch.cuda.synchronize()
    n = deq.shape[1]
    for o in range(0, n, 65536):
        la, lb = a.kernel_launches(), b.kernel_launches()
        a.pushSamplesDevice(ta.data_ptr() + o * 8, 65536, n, fs); a.process()
        b.pushIQDevice(tb.data_ptr() + o * 4, api.IQ_CS16, 65536, n, fs); b.process()
        assert b.kernel_launches() - lb == a.kernel_launches() - la
        _compare(a, b, N_CH, "offset %d" % o)
    _finish(a, b, N_CH)


def test_format_switching_every_call():
    """One handle fed a different format (and host / device entry) every call against one cf32 handle fed the same values:
    the stage-1 carry holds dequantised cf32 whatever format left it."""
    import torch
    fs = 2.048e6
    x = _signals(fs, False)
    n = x.shape[1]
    qs = {f: api.quantise(x, f, SCALE) for f in FORMATS}
    a, b = _pair("f256", N_CH)
    dev = {f: _Dev(torch, N_CH, max(CHUNKS), t, 2) for f, t in
           ((api.IQ_CF32, torch.float32), (api.IQ_CS16, torch.int16), (api.IQ_CS8, torch.int8), (api.IQ_CU8, torch.uint8))}
    dev_a = _Dev(torch, N_CH, max(CHUNKS), torch.float32, 2)
    rot = [api.IQ_CS16, api.IQ_CF32, api.IQ_CU8, api.IQ_CS8]
    for i, (o, k) in enumerate(_chunks(n)):
        f = rot[i % 4]
        on_device = (i // 4) % 2 == 1
        if f == api.IQ_CF32:
            xa = np.ascontiguousarray(x[:, o:o + k])
            xb = xa.view(np.float32)
        else:
            xb = qs[f][:, 2 * o:2 * (o + k)]
            xa = api.dequantise(xb, f)
        if on_device:
            pa, pitch_a = dev_a.put(torch, xa.view(np.float32))
            a.pushSamplesDevice(pa, k, pitch_a, fs); a.process()
            pb, pitch_b = dev[f].put(torch, xb)
            b.pushIQDevice(pb, f, k, pitch_b, fs)
        else:
            a.pushSamplesBatch(np.ascontiguousarray(xa), fs); a.process()
            b.pushIQBatch(xb, f, fs)
        b.process()
        _compare(a, b, N_CH, "call %d format %d" % (i, f))
    _finish(a, b, N_CH)


@pytest.mark.parametrize("entry", ["host", "batch", "device"])
@pytest.mark.parametrize("fmt", [api.IQ_CS16, api.IQ_CU8], ids=lambda f: FMT_ID[f])
def test_per_channel_nco(fmt, entry):
    """NCOs on the channels: host pushes are widened and mixed by K0, a device push is widened and then mixed inside K1 like
    the cf32 device push (fused NCO).  Bitwise equal to the cf32 push with the same NCOs."""
    import torch
    fs = 2.048e6
    x = _signals(fs, False)
    q = api.quantise(x, fmt, SCALE)
    deq = api.dequantise(q, fmt)
    n = deq.shape[1]
    a, b = _pair("f256", N_CH, NCO_HZ)
    ta = torch.from_numpy(deq.view(np.float32)).cuda()
    tb = torch.from_numpy(q).cuda()
    torch.cuda.synchronize()
    for o in range(0, n - n % 65536, 65536):
        k = 65536
        if entry == "host":
            for c in range(N_CH):
                a.pushSamples(c, deq[c, o:o + k], fs); b.pushIQ(c, q[c, 2 * o:2 * (o + k)], fmt, fs)
        elif entry == "batch":
            a.pushSamplesBatch(deq[:, o:o + k], fs); b.pushIQBatch(q[:, 2 * o:2 * (o + k)], fmt, fs)
        else:
            a.pushSamplesDevice(ta.data_ptr() + o * 8, k, n, fs)
            b.pushIQDevice(tb.data_ptr() + o * api.IQ_BYTES[fmt], fmt, k, n, fs)
        a.process(); b.process()
        _compare(a, b, N_CH, "offset %d" % o)
    _finish(a, b, N_CH)


def test_argument_errors():
    import torch
    dec = api.BatchDecoder(2, baud=300.0)
    lib, h = dec._lib, dec._h
    buf = np.zeros(4096, np.int16)
    t = torch.zeros(2 * 4096, dtype=torch.int16, device="cuda")
    p = t.data_ptr()
    for f in (4, -1, 99):                                        # unknown format
        assert lib.hbd_push_iq(h, 0, buf.ctypes.data, f, 16, 2.048e6) == api.HBD_ERR_ARG
        assert lib.hbd_push_iq_batch(h, buf.ctypes.data, f, 16, 16, 2.048e6) == api.HBD_ERR_ARG
        assert lib.hbd_push_iq_device(h, p, f, 16, 16, 2.048e6) == api.HBD_ERR_ARG
        assert lib.hbd_push_iq_wideband(h, buf.ctypes.data, f, 16, 2.048e6) == api.HBD_ERR_ARG
        assert lib.hbd_push_iq_wideband_device(h, p, f, 16, 2.048e6) == api.HBD_ERR_ARG
    assert lib.hbd_push_iq_device(h, p + 4, api.IQ_CS16, 16, 16, 2.048e6) == api.HBD_ERR_ARG      # misaligned rows
    assert lib.hbd_push_iq_device(h, p + 8, api.IQ_CS8, 16, 16, 2.048e6) == api.HBD_ERR_ARG
    assert lib.hbd_push_iq_device(h, p, api.IQ_CS16, 16, 18, 2.048e6) == api.HBD_ERR_ARG          # pitch not a multiple of 4
    assert lib.hbd_push_iq_device(h, p, api.IQ_CS8, 16, 20, 2.048e6) == api.HBD_ERR_ARG           # ... of 8
    assert lib.hbd_push_iq_device(h, p, api.IQ_CU8, 16, 12, 2.048e6) == api.HBD_ERR_ARG           # pitch < n
    assert lib.hbd_push_iq_device(h, p, api.IQ_CS16, 16, 20, 2.048e6) == api.HBD_OK               # aligned: accepted
    assert lib.hbd_push_iq_batch(h, buf.ctypes.data, api.IQ_CS16, 16, 16, 2.048e6) == api.HBD_ERR_STATE   # device push pending
    dec.process()


def _ring_run(torch, q, fmt, n_ch, L, fs, chunk, steps, gather):
    dec = api.BatchDecoder(n_ch, baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    dec.set_stream(torch.cuda.current_stream().cuda_stream)
    bps = api.IQ_BYTES[fmt]
    slices = L // chunk
    if gather:
        dec.dist_init(0, 1, None)
        sink = api.ResultSink(n_ch)
    for i in range(steps):
        dec.pushIQDevice(q.data_ptr() + (i % slices) * chunk * bps, fmt, chunk, L, fs)
        dec.process_async()
        if gather and (i + 1) % 16 == 0:
            dec.collect_ready(4)
            assert dec.gather_results(sink) == n_ch
    dec.collect()
    if not gather:
        return [dec.poll_chars(c) for c in range(n_ch)], [dec.poll_sentences(c) for c in range(n_ch)]
    while True:
        assert dec.gather_results(sink) == n_ch
        if all(not dec.poll_chars(c) for c in (0, n_ch // 2, n_ch - 1)):
            break
    return [sink.poll_chars(c) for c in range(n_ch)], [sink.poll_sentences(c) for c in range(n_ch)]


def _check_ring(oracle_kind, q, fmt, got_chars, got_sents, n_ch, L, fs, chunk, steps):
    for c in range(n_ch):
        want = synth.ring_sentence(c).strip().lstrip("$").encode()
        assert len(got_sents[c]) == 2 and all(s == want for s in got_sents[c]), "channel %d: %r" % (c, got_sents[c])
    cfg = po.make_config(baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=256, record=False)
    bad = []
    for c0 in range(0, n_ch, 256):
        iq = api.dequantise(q[c0:c0 + 256].cpu().numpy(), fmt)
        ref_chars, ref_sents = po.run_ring(oracle_kind, cfg, iq, os.cpu_count() or 4, fs, chunk, 0, steps)
        bad += [c0 + k for k in range(iq.shape[0]) if got_chars[c0 + k] != ref_chars[k] or got_sents[c0 + k] != ref_sents[k]]
    assert not bad, "%d of %d channels differ from the %s oracle, first: %r" % (len(bad), n_ch, oracle_kind, bad[:8])


def _quantised_ring(torch, n_ch, fmt, fs):
    dt = {api.IQ_CS16: torch.int16, api.IQ_CS8: torch.int8, api.IQ_CU8: torch.uint8}[fmt]
    L = synth.ring_length(fs, 300.0)
    q = torch.empty((n_ch, 2 * L), dtype=dt, device="cuda")
    for c0 in range(0, n_ch, 512):                   # generate + quantise in slabs: the cf32 ring never exists whole
        ring = synth.ring_iq_torch(c0, min(512, n_ch - c0), torch.device("cuda", 0), fs, 300.0, snr_db=-15.0)
        q[c0:c0 + ring.shape[0]] = api.quantise(torch.view_as_complex(ring), fmt, SCALE).reshape(ring.shape[0], -1)
        del ring
    torch.cuda.synchronize()
    return q, L


def test_cfg4_full_width_4096_channels_cs16(oracle_kind):
    """BASELINE configs[3] at full size from a CS16 device ring (4096 x 1 638 400 samples, 27 GB) through the native K1:
    pipelined calls, results through the gather path; every channel against the oracle on the dequantised samples."""
    import torch
    fs, chunk, n_ch = 2.048e6, 65536, 4096
    q, L = _quantised_ring(torch, n_ch, api.IQ_CS16, fs)
    steps = 2 * (L // chunk) + 7
    chars, sents = _ring_run(torch, q, api.IQ_CS16, n_ch, L, fs, chunk, steps, gather=True)
    _check_ring(oracle_kind, q, api.IQ_CS16, chars, sents, n_ch, L, fs, chunk, steps)
    del q
    torch.cuda.empty_cache()


def test_ring_256_channels_cu8(oracle_kind):
    import torch
    fs, chunk, n_ch = 2.048e6, 65536, 256
    q, L = _quantised_ring(torch, n_ch, api.IQ_CU8, fs)
    steps = 2 * (L // chunk) + 7
    chars, sents = _ring_run(torch, q, api.IQ_CU8, n_ch, L, fs, chunk, steps, gather=False)
    _check_ring(oracle_kind, q, api.IQ_CU8, chars, sents, n_ch, L, fs, chunk, steps)


def test_example_decodes_a_cu8_file(tmp_path, oracle_kind):
    """examples/decode_cf32_file.cpp on an rtl_sdr-style capture (unsigned 8-bit I, Q): what the reference Decoder makes of
    the dequantised samples, pushed the same way (65 536 samples per call)."""
    fs, baud = 2.048e6, 300.0
    iq, _ = synth.channel_iq(9, 2, fs, baud, snr_db=-12.0)
    q = api.quantise(iq[:len(iq) // 65536 * 65536], api.IQ_CU8, SCALE)
    path = str(tmp_path / "cap.cu8")
    q.tofile(path)
    exe = str(tmp_path / "decode")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    lib_dir = os.path.join(ROOT, "habdec_b200")
    subprocess.run([cxx, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "decode_cf32_file.cpp"),
                    "-L", lib_dir, "-lhabdec_b200", "-Wl,-rpath," + lib_dir, "-o", exe], check=True)
    out = subprocess.run([exe, path, repr(fs), repr(baud), "8", "2", "256", "cu8"], check=True, capture_output=True).stdout.decode("latin1")
    ref = (po.RefDecoder if oracle_kind == "ref" else po.PortDecoder)(po.make_config(baud=baud)).run(api.dequantise(q, api.IQ_CU8), fs)
    sents = [l[len("SENTENCE "):].encode() for l in out.splitlines() if l.startswith("SENTENCE ")]
    assert sents == ref.sentences() and len(sents) >= 1
    assert ("last sentence: " + ref.last_sentence().decode()) in out.splitlines()
