"""Wideband scanner on the GPU (hbd_scanner): the averaged spectrum against the float64 restatement (scan_ref.welch),
its independence of input format and of how a capture is cut into pushes, detection on synthetic captures, and the
loop scan -> NCO per found signal -> channeliser decode, checked against pre-mix + reference Decoder."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import scan_ref
from habdec_b200 import api, synth
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 65536
INT_FMTS = [api.IQ_CS16, api.IQ_CS8, api.IQ_CU8]


def rel_l2(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _test_capture(n, seed, amp=0.25):
    """Complex noise with a few carriers, |I|, |Q| well inside [-1, 1) so that every integer format keeps it."""
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    x = amp * (rng.standard_normal(n) + 1j * rng.standard_normal(n)) / np.sqrt(2.0)
    for f, a in ((0.1234, 0.2), (-0.31, 0.05), (0.4001, 0.01)):
        x += a * np.exp(2j * np.pi * f * t)
    return x.astype(np.complex64)


def _as_fmt(x, fmt):
    """(what the scanner is given, the cf32 values it stands for)"""
    if fmt == api.IQ_CF32:
        return x, x
    q = api.quantise(x, fmt)
    return q, api.dequantise(q, fmt)


def _psd_of(N, pushes, fs=1e6):
    s = api.Scanner(N)
    for arr, fmt in pushes:
        s.push(arr, fs, fmt)
    return s.psd()


def _payload_capture(fs, offsets, bauds, n, snr_db, seed=1, cw=None):
    """RTTY 8N2 payloads (425 Hz shift) at `offsets`, text repeated to fill n samples, full-band SNR snr_db."""
    x = np.zeros(n, dtype=np.complex128)
    for c, (f0, bd) in enumerate(zip(offsets, bauds)):
        text = "".join(synth.make_sentence(c, k) for k in range(4)).encode()
        bits = synth.uart_bits(text, 8, 2, 40, 60)
        x += synth.fsk_iq(bits, fs, bd, 425.0, f0, None, n_samples=n, phase0=0.3 * c)
    if cw is not None:
        x += 0.5 * np.exp(2j * np.pi * cw * np.arange(n) / fs)
    rng = np.random.default_rng(seed)
    sigma = 10.0 ** (-snr_db / 20.0) / np.sqrt(2.0)
    x += sigma * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return x.astype(np.complex64)


# ---- spectrum ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [4096, 65536, 1 << 20])
@pytest.mark.parametrize("fmt", [api.IQ_CF32] + INT_FMTS)
def test_psd_matches_float64_welch(N, fmt):
    n = 5 * N // 2 + N // 3                           # four complete segments and a tail that waits
    given, values = _as_fmt(_test_capture(n, seed=N + fmt), fmt)
    psd, S = _psd_of(N, [(given, fmt)])
    want, S_ref = scan_ref.welch(values, N)
    assert S == S_ref == 4
    assert psd.dtype == np.float32 and psd.shape == (N,)
    assert rel_l2(psd, want) <= 1e-5
    assert int(np.argmax(psd)) == int(np.argmax(want))


@pytest.mark.parametrize("fmt", INT_FMTS)
def test_integer_push_equals_cf32_push_of_dequantised(fmt):
    """Host and device pushes: an integer capture gives bit for bit the PSD of the cf32 push of api.dequantise(...)."""
    import torch
    N, n = 65536, 9 * CHUNK + 12345
    q, deq = _as_fmt(_test_capture(n, seed=40 + fmt), fmt)
    want, S = _psd_of(N, [(deq, api.IQ_CF32)])
    got, S2 = _psd_of(N, [(q, fmt)])
    assert S == S2 and np.array_equal(got, want)
    dq = torch.from_numpy(np.ascontiguousarray(q)).cuda()
    dv = torch.from_numpy(deq.view(np.float32)).cuda()
    torch.cuda.synchronize()
    a, b = api.Scanner(N), api.Scanner(N)
    for o in range(0, n, CHUNK):
        k = min(CHUNK, n - o)
        a.push_device(dq.data_ptr() + o * api.IQ_BYTES[fmt], k, 1e6, fmt)
        b.push_device(dv.data_ptr() + o * 8, k, 1e6)
    pa, sa = a.psd()
    pb, sb = b.psd()
    assert sa == sb == S and np.array_equal(pa, want) and np.array_equal(pb, want)


@pytest.mark.parametrize("N", [4096, 65536])
def test_chunking_invariance(N):
    """One block, 65 536-sample pushes, odd pushes with 1-sample and empty ones, and device pushes: bitwise equal PSDs."""
    import torch
    n = 40 * N // 2 + 777
    x = _test_capture(n, seed=3)
    ref, S = _psd_of(N, [(x, api.IQ_CF32)])
    assert S == (n - N) // (N // 2) + 1
    cuts = [np.arange(0, n, CHUNK)]
    rng = np.random.default_rng(N)
    odd = [0, 1, 0, 1, 3, N - 5, 0, N // 2 + 1, 1]
    while sum(odd) < n:
        odd.append(int(rng.choice([0, 1, 7, 1000, N // 3, 3 * N + 11, 100003])))
    cuts.append(np.cumsum([0] + odd)[:-1])
    for starts in cuts:
        ends = list(starts[1:]) + [n]
        got, S2 = _psd_of(N, [(x[a:min(b, n)], api.IQ_CF32) for a, b in zip(starts, ends) if a <= n])
        assert S2 == S and np.array_equal(got, ref)
    dev = torch.from_numpy(x.view(np.float32)).cuda()
    torch.cuda.synchronize()
    s = api.Scanner(N)
    o = 0
    for k in (N // 2, 2, 6, 3 * N):                # 16-byte aligned starts, well inside the capture
        s.push_device(dev.data_ptr() + o * 8, k, 1e6)
        o += k
    s.push(x[o:], 1e6)                             # the rest from the host
    got, S3 = s.psd()
    assert S3 == S and np.array_equal(got, ref)


def test_before_first_segment_and_reset():
    N = 4096
    s = api.Scanner(N)
    psd, S = s.psd()
    assert S == 0 and not psd.any() and s.find() == []
    x = _test_capture(3 * N, seed=9)
    s.push(x[:N - 1], 2e6)
    psd, S = s.psd()
    assert S == 0 and not psd.any() and s.find() == []
    s.push(x[N - 1:], 2e6)
    assert s.psd()[1] == 5
    lib = api.load()
    assert lib.hbd_scan_push(s._s, x.ctypes.data, api.IQ_CF32, 10, 1e6) == api.HBD_ERR_STATE     # fs change without reset
    s.reset()
    s.push(x[5:], 1e6)                          # after a reset: like a fresh scanner, at a new rate
    fresh, S_f = _psd_of(N, [(x[5:], api.IQ_CF32)], fs=1e6)
    got, S_g = s.psd()
    assert S_g == S_f and np.array_equal(got, fresh)
    assert np.allclose(s.freqs()[[0, N // 2]], [-0.5e6, 0.0])


def test_argument_errors():
    import torch
    lib = api.load()
    h = C.c_void_p()
    for bad in (0, 2048, 4097, 12288, 1 << 21, 3 << 12):
        assert lib.hbd_scanner_create(0, bad, C.byref(h)) == api.HBD_ERR_ARG, bad
    s = api.Scanner(4096)
    x = np.zeros(100, dtype=np.complex64)
    assert lib.hbd_scan_push(s._s, x.ctypes.data, 7, 100, 1e6) == api.HBD_ERR_ARG
    assert lib.hbd_scan_push(s._s, None, api.IQ_CF32, 100, 1e6) == api.HBD_ERR_ARG
    dev = torch.zeros(1024, dtype=torch.float32, device="cuda")
    assert lib.hbd_scan_push_device(s._s, dev.data_ptr() + 8, api.IQ_CF32, 100, 1e6) == api.HBD_ERR_ARG
    assert lib.hbd_scan_push_device(s._s, dev.data_ptr() + 2, api.IQ_CS8, 100, 1e6) == api.HBD_ERR_ARG
    assert lib.hbd_scan_push_device(s._s, dev.data_ptr(), -1, 100, 1e6) == api.HBD_ERR_ARG
    assert lib.hbd_scan_push_device(s._s, dev.data_ptr(), api.IQ_CS16, 100, 1e6) == api.HBD_OK


# ---- detection ----------------------------------------------------------------------------------------------------------
DET_FS, DET_N = 2.5e6, 65536
DET_OFFS, DET_BAUDS = [-900e3, -310e3, -40e3, 55e3, 420e3], [50.0, 100.0, 300.0, 300.0, 100.0]


@pytest.mark.parametrize("snr_db", [-8.0, -28.0])
def test_detection_on_synthetic_capture(snr_db):
    """Five payloads spread over the band (50 / 100 / 300 baud, 425 Hz shift) and a CW carrier, 119 segments: every payload
    within a bin of its centre and two bins of its shift, nothing else (the carrier neither); the GPU spectrum gives the
    same signals as the float64 restatement's."""
    n = 60 * DET_N
    x = _payload_capture(DET_FS, DET_OFFS, DET_BAUDS, n, snr_db, cw=700e3)
    s = api.Scanner(DET_N)
    s.push(x, DET_FS)
    psd, S = s.psd()
    assert S == 119
    bw = DET_FS / DET_N
    found = s.find()
    assert len(found) == len(DET_OFFS), found
    for f, truth in zip(found, DET_OFFS):
        assert abs(f["center_hz"] - truth) <= bw and abs(f["shift_hz"] - 425.0) <= 2 * bw, (f, truth)
        assert f["snr_db"] >= 10.0
    want = scan_ref.detect(scan_ref.welch(x, DET_N)[0].astype(np.float32), DET_FS)
    assert [(f["bin_lo"], f["bin_hi"]) for f in found] == [(w[3], w[4]) for w in want]
    assert api.scan_detect(psd, DET_FS) == found


def test_noise_gives_no_detections():
    rng = np.random.default_rng(2)
    n = 17 * DET_N // 2 + 5
    x = ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) / np.sqrt(2.0)).astype(np.complex64)
    s = api.Scanner(DET_N)
    s.push(x, DET_FS)
    assert s.psd()[1] == 16 and s.find() == []


# ---- end to end: scan, tune, decode -----------------------------------------------------------------------------------
def _short_sentence(c, k=0):
    body = "SCAN%02d,%d,12:00:%02d,%d" % (c, k, c, 700 * c + k)
    return "$$" + body + "*" + synth.crc16_ccitt(body.encode()) + "\n"


def _sentence_capture(fs, offsets, baud, snr_db, seed=7):
    texts = [_short_sentence(c) for c in range(len(offsets))]
    bits = [synth.uart_bits(t.encode(), 8, 2, 30, 40) for t in texts]
    n = (max(int(len(b) * fs / baud) for b in bits) // CHUNK + 1) * CHUNK
    x = np.zeros(n, dtype=np.complex128)
    for c, (b, f) in enumerate(zip(bits, offsets)):
        x += synth.fsk_iq(b, fs, baud, 425.0, f, None, n_samples=n, phase0=0.3 * c)
    rng = np.random.default_rng(seed)
    sigma = 10.0 ** (-snr_db / 20.0) / np.sqrt(2.0)
    x += sigma * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return x.astype(np.complex64), texts


@pytest.mark.parametrize("fs,n_fft,offsets,device", [
    (2.5e6, 65536, [-700e3, -123e3, 310e3, 905e3], False),
    (20e6, 1 << 20, [-7.3e6, 0.6e6, 8.1e6], True),
])
def test_scan_then_decode(oracle_kind, fs, n_fft, offsets, device):
    """Scan the capture, put one decoder channel's NCO on every signal found, push the same capture to the channeliser
    (host, or device on the scanner's stream): characters and sentences equal pre-mix at the found centre + reference."""
    import torch
    baud = 300.0
    x, texts = _sentence_capture(fs, offsets, baud, snr_db=-8.0)
    n = len(x)
    scan = api.Scanner(n_fft)
    if device:
        stream = torch.cuda.current_stream()
        cap = torch.from_numpy(x.view(np.float32)).cuda()
        scan.set_stream(stream.cuda_stream)
        for o in range(0, n, 1 << 22):
            scan.push_device(cap.data_ptr() + o * 8, min(1 << 22, n - o), fs)
    else:
        scan.push(x, fs)
    found = scan.find()
    assert len(found) == len(offsets), found
    centers = [f["center_hz"] for f in found]
    for c, truth in zip(centers, offsets):
        assert abs(c - truth) <= fs / n_fft
    dec = api.BatchDecoder(len(centers), baud=baud, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    if device:
        dec.set_stream(stream.cuda_stream)
    for ch, c in enumerate(centers):
        dec.set_nco(c, ch)
    for o in range(0, n, CHUNK):
        if device:
            dec.pushWidebandDevice(cap.data_ptr() + o * 8, CHUNK, fs)
        else:
            dec.pushWideband(x[o:o + CHUNK], fs)
        dec.process()
    for ch, c in enumerate(centers):
        ref = (po.RefDecoder if oracle_kind == "ref" else po.PortDecoder)(po.make_config(baud=baud, rtty_bits=8, rtty_stops=2.0, dec_factor=256))
        ph = 0.0
        for o in range(0, n, CHUNK):
            mixed, ph = po.premix(x[o:o + CHUNK], fs, c, ph)
            ref.push_process(mixed, fs)
        assert dec.poll_chars(ch) == ref.chars(), "channel %d" % ch
        assert dec.poll_sentences(ch) == ref.sentences() == [texts[ch].strip()[2:].encode()], "channel %d" % ch


def test_cpp_facade_prints_the_python_signals(tmp_path):
    """tests/cpp/scan_find.cpp over include/habdec_b200/Scanner.hpp, fed in 100 000-sample pushes, prints the signals the
    Python Scanner finds in one push."""
    n = 40 * DET_N
    x = _payload_capture(DET_FS, DET_OFFS[1:4], DET_BAUDS[1:4], n, -20.0, seed=5)
    path = str(tmp_path / "cap.cf32")
    x.tofile(path)
    exe = str(tmp_path / "scan_find")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    lib_dir = os.path.join(ROOT, "habdec_b200")
    subprocess.run([cxx, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "scan_find.cpp"),
                    "-L", lib_dir, "-lhabdec_b200", "-Wl,-rpath," + lib_dir, "-lpthread", "-o", exe], check=True)
    out = subprocess.run([exe, path, repr(DET_FS), str(DET_N), "100000"], check=True, capture_output=True, text=True).stdout.splitlines()
    s = api.Scanner(DET_N)
    s.push(x, DET_FS)
    found = s.find()
    assert len(found) == 3
    assert out[0] == "NSEG %d" % s.psd()[1]
    sig = [l.split() for l in out[1:]]
    assert [(float(a[1]), float(a[2]), float(a[3]), int(a[4]), int(a[5])) for a in sig] == \
        [(f["center_hz"], f["shift_hz"], f["snr_db"], f["bin_lo"], f["bin_hi"]) for f in found]
