"""Which route each hbd_push_* entry point takes, pinned by kernel launches.

For each of the ten C entry points (the hbd_push_iq* ones in every format): the return code, the kernel launches of the
push and the kernel launches of the hbd_process after it.  This is done over the first stage of the plan (factor 256:
K1 has the fused NCO and the native integer read; factor 32: it has neither), with and without an NCO, with and without
host samples already staged, and with HBD_NCO_FUSED unset and 0.  Then the state and argument errors of every entry
point.  That the routes compute the same samples is checked bitwise by test_gpu_iq_formats.py and test_gpu_nco.py."""
import os

import numpy as np
import pytest

from habdec_b200 import api

pytestmark = pytest.mark.gpu

N_CH, N, N_STAGED = 3, 8192, 1000
FS = {256: 2.048e6, 32: 256e3}
FMT = {"cf32": api.IQ_CF32, "cs16": api.IQ_CS16, "cs8": api.IQ_CS8, "cu8": api.IQ_CU8}
NCO_CH, NCO_HZ = 0, 20e3   # channel 0 only: a one-channel push to channel 2 then sees an NCO set, but not its own

SHAPE = {"samples": "channel", "samples_batch": "matrix", "samples_device": "matrix", "wideband": "row", "wideband_device": "row",
         "iq": "channel", "iq_batch": "matrix", "iq_device": "matrix", "iq_wideband": "row", "iq_wideband_device": "row"}
CASES = [(e, f, ch) for e in SHAPE for f in (FMT if e.startswith("iq") else ["cf32"])
         for ch in ((0, 2) if SHAPE[e] == "channel" else (None,))]


def _label(case):
    e, f, ch = case
    return "%s.%s%s" % (e, f, "" if ch is None else "/%d" % ch)


def _call(L, h, entry, fmt, ch, p, n, pitch, fs):
    return {
        "samples": lambda: L.hbd_push_samples(h, ch, p, n, fs),
        "samples_batch": lambda: L.hbd_push_samples_batch(h, p, n, pitch, fs),
        "samples_device": lambda: L.hbd_push_samples_device(h, p, n, pitch, fs),
        "wideband": lambda: L.hbd_push_wideband(h, p, n, fs),
        "wideband_device": lambda: L.hbd_push_wideband_device(h, p, n, fs),
        "iq": lambda: L.hbd_push_iq(h, ch, p, fmt, n, fs),
        "iq_batch": lambda: L.hbd_push_iq_batch(h, p, fmt, n, pitch, fs),
        "iq_device": lambda: L.hbd_push_iq_device(h, p, fmt, n, pitch, fs),
        "iq_wideband": lambda: L.hbd_push_iq_wideband(h, p, fmt, n, fs),
        "iq_wideband_device": lambda: L.hbd_push_iq_wideband_device(h, p, fmt, n, fs),
    }[entry]()


class _Src:
    """[N_CH][N] samples of every format, in host memory and in (256-byte aligned) device memory; row pitch N."""
    def __init__(self):
        import torch
        rng = np.random.default_rng(11)
        self.c64 = (0.1 * (rng.standard_normal((N_CH, N)) + 1j * rng.standard_normal((N_CH, N)))).astype(np.complex64)
        self.host = {"cf32": self.c64.view(np.uint8)}
        for f in ("cs16", "cs8", "cu8"):
            self.host[f] = rng.integers(0, 256, size=(N_CH, N * api.IQ_BYTES[FMT[f]]), dtype=np.uint8)
        self.dev = {f: torch.from_numpy(a).cuda() for f, a in self.host.items()}
        torch.cuda.synchronize()

    def ptr(self, fmt, device):
        return self.dev[fmt].data_ptr() if device else self.host[fmt].ctypes.data


@pytest.fixture(scope="module")
def src():
    return _Src()


def _decoder(factor, nco=False, fused0=False):
    old = os.environ.pop("HBD_NCO_FUSED", None)
    if fused0:
        os.environ["HBD_NCO_FUSED"] = "0"   # read by hbd_create
    try:
        d = api.BatchDecoder(N_CH, dec_factor=factor)
    finally:
        os.environ.pop("HBD_NCO_FUSED", None)
        if old is not None:
            os.environ["HBD_NCO_FUSED"] = old
    if nco:
        d.set_nco(NCO_HZ, NCO_CH)
    return d


def _route(src, config, case):
    """'rc/push launches/process launches' of one push on a fresh handle ('-': a rejected push, whose launches are not pinned)"""
    factor, nco, staged, fused0 = config
    entry, fmt, ch = case
    d = _decoder(factor, nco, fused0)
    L, h, fs = d._lib, d._h, FS[factor]
    if staged:
        d.pushSamplesBatch(src.c64[:, :N_STAGED], fs)
    k0 = d.kernel_launches()
    rc = _call(L, h, entry, FMT[fmt], ch, src.ptr(fmt, entry.endswith("_device")), N, N, fs)
    k1 = d.kernel_launches()
    assert L.hbd_process(h) == api.HBD_OK
    k2 = d.kernel_launches()
    d.close()
    return "%d/%s/%d" % (rc, k1 - k0 if rc == api.HBD_OK else "-", k2 - k1)


def _config_label(c):
    factor, nco, staged, fused0 = c
    return "%d%s%s%s" % (factor, "N" if nco else "-", "S" if staged else "-", "0" if fused0 else "-")


CONFIGS = [(f, nco, st, f0) for f in (256, 32) for nco in (False, True) for st in (False, True) for f0 in (False, True)]

# Columns: first-stage factor, N: an NCO is set, S: host samples are staged before the push, 0: HBD_NCO_FUSED=0.
# Entries: return code / kernel launches of the push / kernel launches of the following hbd_process.
ROUTES = """
case                     256--- 256--0 256-S- 256-S0 256N-- 256N-0 256NS- 256NS0 32---  32--0  32-S-  32-S0  32N--  32N-0  32NS-  32NS0
samples.cf32/0           0/0/3  0/0/3  0/0/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3  0/0/3  0/0/3  0/0/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3
samples.cf32/2           0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3
samples_batch.cf32       0/0/3  0/0/3  0/0/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3  0/0/3  0/0/3  0/0/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3
samples_device.cf32      0/0/3  0/0/3  -3/-/3 -3/-/3 0/0/3  0/1/3  0/1/3  0/1/3  0/0/3  0/0/3  -3/-/3 -3/-/3 0/1/3  0/1/3  0/1/3  0/1/3
wideband.cf32            0/0/3  0/1/3  0/1/3  0/1/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
wideband_device.cf32     0/0/3  0/1/3  0/1/3  0/1/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq.cf32/0                0/0/3  0/0/3  0/0/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3  0/0/3  0/0/3  0/0/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3
iq.cf32/2                0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3  0/0/3
iq.cs16/0                0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq.cs16/2                0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq.cs8/0                 0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq.cs8/2                 0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq.cu8/0                 0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq.cu8/2                 0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq_batch.cf32            0/0/3  0/0/3  0/0/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3  0/0/3  0/0/3  0/0/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3
iq_batch.cs16            0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq_batch.cs8             0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq_batch.cu8             0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq_device.cf32           0/0/3  0/0/3  -3/-/3 -3/-/3 0/0/3  0/1/3  0/1/3  0/1/3  0/0/3  0/0/3  -3/-/3 -3/-/3 0/1/3  0/1/3  0/1/3  0/1/3
iq_device.cs16           0/0/3  0/0/3  -3/-/3 -3/-/3 0/1/3  0/2/3  0/2/3  0/2/3  0/1/3  0/1/3  -3/-/3 -3/-/3 0/2/3  0/2/3  0/2/3  0/2/3
iq_device.cs8            0/0/3  0/0/3  -3/-/3 -3/-/3 0/1/3  0/2/3  0/2/3  0/2/3  0/1/3  0/1/3  -3/-/3 -3/-/3 0/2/3  0/2/3  0/2/3  0/2/3
iq_device.cu8            0/0/3  0/0/3  -3/-/3 -3/-/3 0/1/3  0/2/3  0/2/3  0/2/3  0/1/3  0/1/3  -3/-/3 -3/-/3 0/2/3  0/2/3  0/2/3  0/2/3
iq_wideband.cf32         0/0/3  0/1/3  0/1/3  0/1/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq_wideband.cs16         0/1/3  0/2/3  0/2/3  0/2/3  0/1/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3
iq_wideband.cs8          0/1/3  0/2/3  0/2/3  0/2/3  0/1/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3
iq_wideband.cu8          0/1/3  0/2/3  0/2/3  0/2/3  0/1/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3
iq_wideband_device.cf32  0/0/3  0/1/3  0/1/3  0/1/3  0/0/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3  0/1/3
iq_wideband_device.cs16  0/1/3  0/2/3  0/2/3  0/2/3  0/1/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3
iq_wideband_device.cs8   0/1/3  0/2/3  0/2/3  0/2/3  0/1/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3
iq_wideband_device.cu8   0/1/3  0/2/3  0/2/3  0/2/3  0/1/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3  0/2/3
"""


def _expected():
    lines = [l.split() for l in ROUTES.strip().splitlines()]
    cols = lines[0][1:]
    return {(row[0], col): v for row in lines[1:] for col, v in zip(cols, row[1:])}


@pytest.mark.parametrize("config", CONFIGS, ids=_config_label)
def test_push_routes(src, config):
    want = _expected()
    col = _config_label(config)
    got = {_label(c): _route(src, config, c) for c in CASES}
    bad = ["%-28s got %-10s want %s" % (k, v, want.get((k, col))) for k, v in got.items() if want.get((k, col)) != v]
    assert not bad, "routes of %s changed:\n%s" % (col, "\n".join(bad))


def _state_message(case, nco):
    """what a matrix / row push with unequal queue depths is told"""
    entry = case[0]
    if SHAPE[entry] == "row":
        return "wideband push needs equal queue depth in all channels"
    if entry.endswith("_device") and not nco:
        return "host push pending"
    return "batch push needs equal queue depth in all channels"


@pytest.mark.parametrize("case", CASES, ids=_label)
def test_state_errors(src, case):
    entry, fmt, ch = case
    device = entry.endswith("_device")

    def push(d, factor):
        return _call(d._lib, d._h, entry, FMT[fmt], ch, src.ptr(fmt, device), N, N, FS[factor])

    def last_error(d):
        return (d._lib.hbd_last_error(d._h) or b"").decode()

    # a device push is pending until the next process
    d = _decoder(256)
    assert d._lib.hbd_push_samples_device(d._h, src.ptr("cf32", True), N, N, FS[256]) == api.HBD_OK
    assert push(d, 256) == api.HBD_ERR_STATE and last_error(d) == "device push pending"
    d.close()

    # unequal queue depths after a one-channel push
    for nco in (False, True):
        d = _decoder(256, nco)
        d.pushSamples(0, src.c64[0, :100], FS[256])
        rc = push(d, 256)
        if SHAPE[entry] == "channel":
            assert rc == api.HBD_OK, last_error(d)
        else:
            assert rc == api.HBD_ERR_STATE and last_error(d) == _state_message(case, nco)
        d.close()

    # a device matrix without an NCO is read in place: nothing may be staged (cf32, native integer K1 at factor 256,
    # integer widened first at factor 32)
    if SHAPE[entry] == "matrix" and device:
        for factor in (256, 32):
            d = _decoder(factor)
            d.pushSamplesBatch(src.c64[:, :100], FS[factor])
            assert push(d, factor) == api.HBD_ERR_STATE and last_error(d) == "host push pending"
            d.close()


@pytest.mark.parametrize("case", CASES, ids=_label)
def test_argument_errors(src, case):
    entry, fmt, ch = case
    shape, device = SHAPE[entry], entry.endswith("_device")
    b = api.IQ_BYTES[FMT[fmt]]
    d = _decoder(256)
    L = d._lib
    p0 = src.ptr(fmt, device)

    def push(h=d._h, p=p0, n=N, pitch=N, c=0 if ch is None else ch, f=FMT[fmt]):
        return _call(L, h, entry, f, c, p, n, pitch, FS[256])

    k0 = d.kernel_launches()
    bad = {"null handle": push(h=None), "null samples": push(p=None)}
    if shape == "channel":
        bad.update({"channel -1": push(c=-1), "channel N_CH": push(c=N_CH)})
    if shape == "matrix":
        bad["pitch < n"] = push(pitch=N - 1)
    if shape == "matrix" and device:
        bad.update({"row not 16-byte aligned": push(p=p0 + 8), "pitch not 16 bytes": push(pitch=N + 8 // b)})
    if entry.startswith("iq"):
        bad["unknown format"] = push(f=7)
    assert {k: v for k, v in bad.items() if v != api.HBD_ERR_ARG} == {}
    assert d.kernel_launches() == k0
    # no samples and no pointer: fine, except for a device matrix
    assert push(p=None, n=0) == (api.HBD_ERR_ARG if shape == "matrix" and device else api.HBD_OK)
    d.close()
