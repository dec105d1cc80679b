"""Handles own their CUDA resources: destroying a decoder or scanner with every optional buffer switched on gives all of
its device memory back, and an allocation the device refuses leaves the handle as it was."""
import ctypes as C
import os

import numpy as np
import pytest

from habdec_b200 import api, synth

pytestmark = pytest.mark.gpu

FS, BAUD, N_CH = 2.048e6, 300.0, 4


def process_device_memory():
    """Device memory NVML accounts to this process (summed over the GPUs), or None if NVML does not list it: the GPU is
    shared, so a device-wide figure would include other users' work."""
    pynvml = pytest.importorskip("pynvml")
    pynvml.nvmlInit()
    try:
        pid, total, seen = os.getpid(), 0, False
        for i in range(pynvml.nvmlDeviceGetCount()):
            for p in pynvml.nvmlDeviceGetComputeRunningProcesses(pynvml.nvmlDeviceGetHandleByIndex(i)):
                if p.pid == pid and p.usedGpuMemory is not None:
                    total += p.usedGpuMemory; seen = True
        return total if seen else None
    finally:
        pynvml.nvmlShutdown()


def use_everything(wide_dev, n_wide):
    """A decoder with every optional buffer allocated, and a scanner."""
    rng = np.random.default_rng(7)
    dec = api.BatchDecoder(N_CH, baud=BAUD, record=True, fft_bins=16384)
    dec.set_ssdv(True)
    dec.set_stats_snapshot(True)
    dec.set_demod_accumulate(True)
    dec.set_kernel_timing(2)
    ints = rng.integers(-2000, 2000, size=(N_CH, 2 * 65536), dtype=np.int16)
    dec.pushIQBatch(ints, api.IQ_CS16, FS)                     # host integers: the upload buffer
    dec.process()
    dec.set_nco(1000.0)
    dec.pushWidebandDevice(wide_dev, n_wide, FS)               # device row through the NCOs: the fused-NCO ring
    dec.process()
    assert dec.setupDecimationStagesBW(600.0) == 4096          # cascaded plan: middle-stage buffers
    iq = (rng.standard_normal((N_CH, 300000)) + 1j * rng.standard_normal((N_CH, 300000))).astype(np.complex64)
    dec.pushSamplesBatch(iq, FS)
    dec.process()
    dec.demod_frames(256, 1)                                  # frame buffer
    sc = api.Scanner(65536)
    sc.push(iq[0], FS)
    sc.psd()
    return dec, sc


def test_destroy_releases_everything():
    torch = pytest.importorskip("torch")
    n_wide = 131072
    wide = torch.zeros(2 * n_wide, dtype=torch.float32, device="cuda")   # allocated once, outside the measured cycles
    torch.cuda.synchronize()
    after = []
    for _ in range(3):
        dec, sc = use_everything(wide.data_ptr(), n_wide)
        dec.close(); sc.close()
        after.append(process_device_memory())
    if after[0] is None:
        pytest.skip("NVML does not list this process (PID namespace)")
    assert after[2] == after[0], "device memory after each destroy (bytes): %r" % after


def decode(dec, iq):
    for o in range(0, iq.shape[1], 65536):
        dec.pushSamplesBatch(np.ascontiguousarray(iq[:, o:o + 65536]), FS)
        dec.process()
    stages = [[dec.debug_stage(c, s).tobytes() for s in (api.STAGE_DECIMATED, api.STAGE_FILTERED, api.STAGE_DEMOD, api.STAGE_PENDING,
                                                         api.STAGE_BITS)] for c in range(N_CH)]
    return [dec.poll_chars(c) for c in range(N_CH)], stages


def test_failed_allocation_leaves_handle_usable():
    sigs = [synth.channel_iq(30 + c, 2, FS, BAUD, snr_db=-12.0)[0] for c in range(N_CH)]
    n = min(len(s) for s in sigs) // 65536 * 65536
    iq = np.stack([s[:n] for s in sigs]).astype(np.complex64)
    hit, twin = api.BatchDecoder(N_CH, baud=BAUD, record=True), api.BatchDecoder(N_CH, baud=BAUD, record=True)
    # a staging matrix of N_CH x 2^33 cf32 samples (256 GiB) is more than the device has: cudaMalloc refuses it before any
    # copy, so the host buffer behind the pointer is never read
    big = 1 << 33
    launches = hit.kernel_launches()
    rc = hit._lib.hbd_push_samples_batch(hit._h, iq.ctypes.data, big, big, C.c_double(FS))
    assert rc == api.HBD_ERR_CUDA
    assert hit.kernel_launches() == launches
    got, want = decode(hit, iq), decode(twin, iq)
    assert got[1] == want[1]
    assert got[0] == want[0] and all(len(x) > 10 for x in got[0])
