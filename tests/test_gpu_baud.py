"""Baud-rate estimation on the GPU (hbd_set_baud_estimation ...): histograms and estimates bit for bit equal to the numpy
restatement (tests/baud_ref.py) on the GPU's own discriminator samples, the rates it finds, applying them, and that it
only observes."""
import math
import os
import subprocess

import numpy as np
import pytest

import baud_ref
from habdec_b200 import api, synth
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 65536
FS3 = 2.048e6          # configs[3] geometry: factor 256, fs_dec 8 kHz
WRONG = 45.45


def sigma_for(fs, snr_inband_db):
    """Per-component noise sigma for a unit-power signal at the given SNR in 3 kHz."""
    full = snr_inband_db - 10.0 * math.log10(fs / 3000.0)
    return 10.0 ** (-full / 20.0) / math.sqrt(2.0)


def sentence(tag, c, k=0):
    body = "%s%02d,%d,12:00:%02d,%d" % (tag, c, k, c, 700 * c + k)
    return "$$" + body + "*" + synth.crc16_ccitt(body.encode()) + "\n"


class Keyer:
    """Continuous-phase 2-FSK of `bits` (repeated without end) at offset f_off, plus noise, generated chunk by chunk."""

    def __init__(self, bits, fs, baud, f_off=0.0, sigma=0.0, seed=0, phase0=0.0, shift=425.0):
        self.bits, self.fs, self.baud, self.f_off, self.sigma, self.shift = bits, fs, baud, f_off, sigma, shift
        self.pos, self.ph = 0, phase0
        self.rng = np.random.default_rng(seed)

    def next(self, n):
        i = ((self.pos + np.arange(n, dtype=np.float64)) * (self.baud / self.fs)).astype(np.int64) % len(self.bits)
        f = np.where(self.bits[i] > 0, 0.5 * self.shift, -0.5 * self.shift) + self.f_off
        ph = self.ph + np.cumsum(2.0 * np.pi * f / self.fs)
        self.ph = float(ph[-1]) % (2.0 * np.pi) if n else self.ph
        self.pos += n
        x = np.exp(1j * ph)
        if self.sigma:
            x = x + self.sigma * (self.rng.standard_normal(n) + 1j * self.rng.standard_normal(n))
        return x


class Silence:
    """Noise only (sigma 0: zeros)."""

    def __init__(self, sigma=0.0, seed=0):
        self.sigma, self.rng = sigma, np.random.default_rng(seed)

    def next(self, n):
        x = np.zeros(n, np.complex128)
        if self.sigma:
            x = x + self.sigma * (self.rng.standard_normal(n) + 1j * self.rng.standard_normal(n))
        return x


def payload_bits(c, nbits, nstops, n_sent=4):
    return synth.uart_bits("".join(synth.make_sentence(c, k) for k in range(n_sent)).encode(), nbits, nstops, 2, 2)


def fields(e):
    return (float(e["baud"]), float(e["nominal"]), float(e["confidence"]), int(e["runs"]), int(e["long_runs"]))


def ref_fields(r):
    return (r["baud"], r["nominal"], r["confidence"], r["runs"], r["long_runs"])


# ---- 1. bit-exact against the restatement -----------------------------------------------------------------------------
SIGS = [(50, 8, 2, 20), (75, 7, 1, 10), (100, 8, 1, 6), (150, 8, 2, 10), (300, 7, 1, 20), (600, 8, 1, 10), (300, 8, 2, 6),
        (600, 7, 1, 20), (50, 7, 1, 10), (100, 8, 2, 20), (150, 7, 1, 6), (75, 8, 1, 20), (300, 8, 1, 10), (600, 8, 2, 6)]


def test_histograms_and_estimates_equal_the_restatement():
    n_ch = len(SIGS) + 2        # + a noise-only and a silent channel
    keyers = [Keyer(payload_bits(c, nb, ns), FS3, b, 0.0, sigma_for(FS3, snr), seed=c, phase0=0.1 * c) for c, (b, nb, ns, snr) in enumerate(SIGS)]
    keyers += [Silence(sigma_for(FS3, 10.0), seed=99), Silence()]
    dec = api.BatchDecoder(n_ch, baud=WRONG, rtty_bits=8, rtty_stops=2.0, dec_factor=256, record=True)
    dec.set_baud_estimation(True)               # before the first push: the rows are sized by the first call
    streams = [[] for _ in range(n_ch)]
    rng = np.random.default_rng(3)
    sizes = [65536, 65536, 40000, 90001, 100, 0, 255, 70000]
    n_small = 0
    for k in range(70):
        if k == 20:
            dec.process()                       # nothing queued at all
        else:
            for c in range(n_ch):
                n = int(rng.choice(sizes)) if k % 3 else 65536
                if n:
                    dec.pushSamples(c, keyers[c].next(n).astype(np.complex64), FS3)
            dec.process()
        n_small += sum(len(dec.debug_stage(c, api.STAGE_DEMOD)) == 0 for c in range(n_ch))
        for c in range(n_ch):
            streams[c].append(dec.debug_stage(c, api.STAGE_DEMOD))
    assert n_small > 0                          # some channels sat out calls in which others worked
    fs = dec.getDecimatedSamplingRate()
    assert fs == 8000.0
    est = dec.baud_estimates()
    for c in range(n_ch):
        d = np.concatenate(streams[c])
        H, long_runs = baud_ref.histogram(d, fs)
        assert np.array_equal(dec.baud_histogram(c), H), "channel %d" % c
        assert fields(est[c]) == ref_fields(baud_ref.score(H, long_runs, fs)), "channel %d" % c
    assert est[n_ch - 1]["runs"] == 0 and fields(est[n_ch - 1])[:3] == (0.0, 0.0, 0.0)
    assert all(est[c]["runs"] > 20 for c in range(len(SIGS)))


# ---- 2. it finds the rate -------------------------------------------------------------------------------------------
RATES = [50, 75, 100, 150, 200, 300, 600]


def _run_batch(dec, keyers, calls, fs=FS3):
    for _ in range(calls):
        dec.pushSamplesBatch(np.stack([k.next(CHUNK) for k in keyers]).astype(np.complex64), fs)
        dec.process()


def test_finds_the_rate_at_configs3_geometry():
    sigs = [(b, nb, ns) for b in RATES for nb, ns in ((8, 2), (7, 1))] + [(297.0, 8, 2)]
    keyers = [Keyer(payload_bits(c, nb, ns), FS3, b, 0.0, sigma_for(FS3, 10.0), seed=c, phase0=0.2 * c) for c, (b, nb, ns) in enumerate(sigs)]
    keyers += [Silence(sigma_for(FS3, 10.0), seed=100 + i) for i in range(2)]
    dec = api.BatchDecoder(len(keyers), baud=WRONG, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    dec.set_baud_estimation(True)
    _run_batch(dec, keyers, int(6.0 * FS3) // CHUNK)
    est = dec.baud_estimates()
    for c, (b, nb, ns) in enumerate(sigs):
        e = est[c]
        assert e["runs"] >= 100, (b, nb, ns, e)
        if b == 297.0:
            assert e["nominal"] == 300.0 and abs(e["baud"] - 297.0) / 297.0 <= 0.003, e
        else:
            assert e["nominal"] == b and e["confidence"] >= 0.8 and abs(e["baud"] - b) / b <= 0.005, (b, nb, ns, e)
    for c in range(len(sigs), len(keyers)):
        assert est[c]["confidence"] < 0.5, est[c]
    applied = dec.apply_baud_estimates()
    assert list(applied[:len(sigs)]) == [300.0 if b == 297.0 else float(b) for b, _, _ in sigs]
    assert not applied[len(sigs):].any()
    assert [dec._lib.hbd_get_baud(dec._h, c) for c in range(len(keyers))] == list(applied[:len(sigs)]) + [WRONG, WRONG]


def test_finds_the_rate_at_configs4_geometry():
    """20 MS/s wideband device pushes through the channels' NCOs, fs_dec = 78 125 Hz."""
    import torch
    fs, chunk = 20e6, 262144
    sigs = [(50, 8, 2, -3.1e6), (300, 7, 1, 1.2e6), (600, 8, 2, 5.3e6)]
    keyers = [Keyer(payload_bits(c, nb, ns), fs, b, f, 0.0, phase0=0.5 * c) for c, (b, nb, ns, f) in enumerate(sigs)]
    noise = Silence(sigma_for(fs, 10.0), seed=5)
    offsets = [f for *_, f in sigs] + [-7.7e6]           # the last channel sees noise only
    dec = api.BatchDecoder(len(offsets), baud=WRONG, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    for c, f in enumerate(offsets):
        dec.set_nco(f, c)
    dec.set_baud_estimation(True)
    buf = torch.empty((chunk, 2), dtype=torch.float32, device="cuda")
    for _ in range(int(6.0 * fs) // chunk):
        x = noise.next(chunk)
        for k in keyers:
            x += k.next(chunk)
        buf.copy_(torch.from_numpy(x.astype(np.complex64).view(np.float32).reshape(chunk, 2)))
        torch.cuda.synchronize()
        dec.pushWidebandDevice(buf.data_ptr(), chunk, fs)
        dec.process()
    assert dec.getDecimatedSamplingRate() == 78125.0
    est = dec.baud_estimates()
    for c, (b, *_rest) in enumerate(sigs):
        e = est[c]
        assert e["runs"] >= 100 and e["nominal"] == b and e["confidence"] >= 0.8 and abs(e["baud"] - b) / b <= 0.005, (b, e)
    assert est[3]["confidence"] < 0.5, est[3]
    applied = dec.apply_baud_estimates()
    assert list(applied) == [50.0, 300.0, 600.0, 0.0]


# ---- 3. apply, then decode exactly like the reference ---------------------------------------------------------------
def test_apply_then_decode_like_the_reference(oracle_kind):
    sigs = [(150, 8, 2), (300, 7, 1), (600, 8, 2)]
    keyers = [Keyer(payload_bits(c, nb, ns, 3), FS3, b, 0.0, sigma_for(FS3, 20.0), seed=10 + c, phase0=0.3 * c) for c, (b, nb, ns) in enumerate(sigs)]
    n_calls, K = 300, 70
    dec = api.BatchDecoder(len(sigs), baud=WRONG, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    for c, (_, nb, ns) in enumerate(sigs):
        dec.rtty_bits(nb, c); dec.rtty_stops(ns, c)
    dec.set_baud_estimation(True)
    refs = [(po.RefDecoder if oracle_kind == "ref" else po.PortDecoder)(po.make_config(baud=WRONG, rtty_bits=nb, rtty_stops=float(ns), dec_factor=256))
            for _, nb, ns in sigs]
    before = []
    for k in range(n_calls):
        x = np.stack([kr.next(CHUNK) for kr in keyers]).astype(np.complex64)
        dec.pushSamplesBatch(x, FS3)
        dec.process()
        for c, r in enumerate(refs):
            r.push_process(x[c], FS3)
        if k == K:
            applied = dec.apply_baud_estimates()
            assert list(applied) == [float(b) for b, _, _ in sigs]
            for c, r in enumerate(refs):
                r.set_param("baud", applied[c])
            before = [len(r.sentences()) for r in refs]
    for c, r in enumerate(refs):
        assert dec.poll_chars(c) == r.chars(), "channel %d" % c
        got = dec.poll_sentences(c)
        assert got == r.sentences(), "channel %d" % c
        assert len(got) > before[c], "channel %d: no sentence after the rate was applied" % c


# ---- 4. an unattended receiver, end to end ----------------------------------------------------------------------------
def test_unattended_receiver():
    fs, chunk, n_fft = 2.5e6, 262144, 65536
    pays = [(50.0, -700e3), (100.0, 210e3), (300.0, 905e3)]
    texts = [[sentence("UR%d" % int(b), i, k) for k in range(4)] for i, (b, _) in enumerate(pays)]
    keyers = [Keyer(synth.uart_bits("".join(t).encode(), 8, 2, 20, 0), fs, b, f, 0.0, phase0=0.4 * i) for i, ((b, f), t) in enumerate(zip(pays, texts))]
    noise = Silence(10.0 ** (8.0 / 20.0) / math.sqrt(2.0), seed=21)      # full-band SNR -8 dB

    def chunk_iq():
        x = noise.next(chunk)
        for k in keyers:
            x += k.next(chunk)
        return x.astype(np.complex64)

    scan = api.Scanner(n_fft)
    first = [chunk_iq() for _ in range(8)]
    for x in first:
        scan.push(x, fs)
    found = scan.find()
    assert len(found) == len(pays), found
    dec = api.BatchDecoder(len(found) + 1, rtty_bits=8, rtty_stops=2.0, dec_factor=256)   # the constructor's default baud
    for ch, f in enumerate(found):
        assert abs(f["center_hz"] - pays[ch][1]) <= fs / n_fft
        dec.set_nco(f["center_hz"], ch)
    dec.set_baud_estimation(True)
    n_calls, k_apply = int(22.0 * fs) // chunk, int(6.5 * fs) // chunk
    polled = [[] for _ in pays]
    for k in range(n_calls):
        dec.pushWideband(first[k] if k < len(first) else chunk_iq(), fs)
        dec.process()
        if k == k_apply:
            applied = dec.apply_baud_estimates()
            assert list(applied) == [50.0, 100.0, 0.0, 0.0]       # the 300-baud channel already had its rate
            polled = [dec.poll_sentences(ch) for ch in range(len(pays))]
    for ch in range(len(pays)):
        after = dec.poll_sentences(ch)
        valid = {t.strip()[2:].encode() for t in texts[ch]}
        assert set(polled[ch] + after) <= valid, (ch, polled[ch], after)
        assert after, "payload %d: no sentence after apply" % ch


# ---- 5. it only observes ----------------------------------------------------------------------------------------------
def test_estimation_only_observes():
    sigs = [(300, 8, 2), (600, 7, 1), (150, 8, 2)]
    n_calls = 40
    keyers = [Keyer(payload_bits(c, nb, ns), FS3, b, 0.0, sigma_for(FS3, 15.0), seed=c) for c, (b, nb, ns) in enumerate(sigs)]
    keyers.append(Silence(sigma_for(FS3, 15.0), seed=9))
    x = np.stack([k.next(n_calls * CHUNK) for k in keyers]).astype(np.complex64)
    decs = [api.BatchDecoder(len(keyers), baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=256) for _ in range(2)]
    decs[0].set_baud_estimation(True)
    l0 = [d.kernel_launches() for d in decs]
    working = 0
    for k in range(n_calls):
        for d in decs:
            if k == 10:
                d.process()                      # nothing queued: no work, no histogram kernel
            elif k == 11:                        # one channel below the decimation factor, the others working
                for c in range(len(keyers)):
                    d.pushSamples(c, x[c, k * CHUNK:k * CHUNK + (100 if c == 1 else CHUNK)], FS3)
                d.process()
            else:
                d.pushSamplesBatch(np.ascontiguousarray(x[:, k * CHUNK:(k + 1) * CHUNK]), FS3)
                d.process()
        working += k != 10
    on, off = (d.kernel_launches() - l for d, l in zip(decs, l0))
    assert on - off == working
    for c in range(len(keyers)):
        assert decs[0].poll_chars(c) == decs[1].poll_chars(c)
        assert decs[0].poll_sentences(c) == decs[1].poll_sentences(c)
    assert np.array_equal(decs[0].stats_all(), decs[1].stats_all())


# ---- 6. life cycle ----------------------------------------------------------------------------------------------------
def test_life_cycle():
    lib = api.load()
    sigs = [(300, 8, 2), (600, 8, 2), (150, 7, 1), (100, 8, 2)]
    keyers = [Keyer(payload_bits(c, nb, ns), FS3, b, 0.0, sigma_for(FS3, 15.0), seed=c) for c, (b, nb, ns) in enumerate(sigs)]
    dec = api.BatchDecoder(len(sigs), baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    h = dec._h
    est = (api.BaudEstimate * len(sigs))()
    assert lib.hbd_get_baud_estimates(h, est, len(sigs)) == api.HBD_ERR_STATE
    assert lib.hbd_apply_baud_estimates(h, 0.8, 100, None) == api.HBD_ERR_STATE
    assert dec.baud_histogram(0).size == 0
    _run_batch(dec, keyers, 5)
    dec.set_baud_estimation(True)               # the rate is known: rows now
    assert dec.baud_histogram(0).size == 1041 and not dec.baud_histogram(0).any()
    _run_batch(dec, keyers, 30)
    H = [dec.baud_histogram(c) for c in range(len(sigs))]
    assert all(x.sum() > 20 for x in H)
    # setters other than the plan leave it alone
    dec.baud(100.0, 0); dec.lowpass_bw(1400.0); dec.set_nco(0.0, 1); dec.set_fft_size(16384); dec.rtty_bits(7, 2)
    assert all(np.array_equal(dec.baud_histogram(c), H[c]) for c in range(len(sigs)))
    dec.reset_channels([1, 2])
    assert not dec.baud_histogram(1).any() and not dec.baud_histogram(2).any()
    assert np.array_equal(dec.baud_histogram(0), H[0]) and np.array_equal(dec.baud_histogram(3), H[3])
    e = dec.baud_estimates()
    assert e[1]["runs"] == e[2]["runs"] == e[1]["long_runs"] == 0 and e[0]["runs"] == H[0].sum()
    _run_batch(dec, keyers, 10)
    assert dec.baud_histogram(1).any()
    # a plan change restarts every channel; a new fs_dec resizes the histogram
    assert dec.setupDecimationStagesFactor(256) == 256
    assert all(not dec.baud_histogram(c).any() for c in range(len(sigs)))
    assert dec.setupDecimationStagesFactor(128) == 128
    assert dec.baud_histogram(0).size == baud_ref.geometry(16000.0)[0] + 1
    _run_batch(dec, keyers, 10)
    assert dec.baud_histogram(0).any()
    # off, then on: restarted
    dec.set_baud_estimation(False)
    assert dec.baud_histogram(0).size == 0
    assert lib.hbd_get_baud_estimates(h, est, len(sigs)) == api.HBD_ERR_STATE
    dec.set_baud_estimation(True)
    assert all(not dec.baud_histogram(c).any() for c in range(len(sigs)))
    assert all(r["runs"] == 0 for r in dec.baud_estimates())
    buf = np.zeros(4, np.uint32)
    assert lib.hbd_get_baud_histogram(h, -1, buf.ctypes.data, 4) == 0
    assert lib.hbd_get_baud_histogram(h, len(sigs), buf.ctypes.data, 4) == 0
    assert lib.hbd_get_baud_estimates(h, est, len(sigs)) == len(sigs)


# ---- 7. C++ facade ----------------------------------------------------------------------------------------------------
def test_cpp_facade_equals_python(tmp_path):
    sigs = [(300, 8, 2), (600, 8, 2)]
    n_calls = 40
    keyers = [Keyer(payload_bits(c, nb, ns), FS3, b, 0.0, sigma_for(FS3, 20.0), seed=c) for c, (b, nb, ns) in enumerate(sigs)]
    x = np.stack([k.next(n_calls * CHUNK) for k in keyers]).astype(np.complex64)
    path = str(tmp_path / "batch.cf32")
    x.tofile(path)
    exe = str(tmp_path / "baud_facade")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    lib_dir = os.path.join(ROOT, "habdec_b200")
    subprocess.run([cxx, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "baud_facade.cpp"),
                    "-L", lib_dir, "-lhabdec_b200", "-Wl,-rpath," + lib_dir, "-lpthread", "-o", exe], check=True)
    out = subprocess.run([exe, path, str(len(sigs)), str(n_calls * CHUNK), repr(FS3)], check=True, capture_output=True, text=True).stdout
    dec = api.BatchDecoder(len(sigs), baud=WRONG, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    dec.set_baud_estimation(True)
    for k in range(n_calls):
        dec.pushSamplesBatch(np.ascontiguousarray(x[:, k * CHUNK:(k + 1) * CHUNK]), FS3)
        dec.process()
    est = dec.baud_estimates()
    applied = dec.apply_baud_estimates(0.8, 50)
    want = "".join("EST%d %r %r %r %d %d\n" % ((c,) + fields(est[c])) for c in range(len(sigs)))
    want += "APPLIED %d\n" % int((applied != 0).sum())
    want += "".join("BAUD%d %r\n" % (c, dec._lib.hbd_get_baud(dec._h, c)) for c in range(len(sigs)))
    got = [ln.split(" ") for ln in out.splitlines()]
    assert [[w[0]] + [float(v) for v in w[1:]] for w in got] == [[w[0]] + [float(v) for v in w[1:]] for w in (ln.split(" ") for ln in want.splitlines())]
    assert int((applied != 0).sum()) == 2
