"""Wideband scanner (hbd_scanner, N = 2^20) on one GPU, two measurements in one process:

1. standalone: a device-resident capture of 4 GiB (cf32: 2^29 samples; CS8: 2^31 samples), larger than L2, pushed in
   2^22-sample device pushes.  Capture GS/s and scan time per segment from CUDA events around whole passes, against two
   bounds: FP32 (2 (5 log2 N + 10) flop per input sample at 50 % overlap, over 148 SMs x 128 FMA/clk at the card's
   maximum SM clock -- a computed peak, not a measured one) and HBM (input bytes per sample, over the device copy
   bandwidth measured here; a second figure adds the 32 B per sample the pass-A -> pass-B intermediate would cost if it
   left L2).  Formats alternate over the repeats.
2. beside the channeliser: BASELINE configs[4] (1024 NCO channels, 20 MS/s, 65 536-sample device pushes of one capture,
   as tools/bench_wideband.py) with and without the scanner reading the same slices on the same stream; the two legs
   alternate within the session, the spread over repeats is reported.

Writes profiles/r4_scan.json (or --out).
    python tools/bench_scan.py [--repeats 5] [--steps 200] [--out profiles/r4_scan.json]
"""
from __future__ import annotations

import argparse
import gc
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_FFT, PUSH, FS, CHUNK, N_CH = 1 << 20, 1 << 22, 20e6, 65536, 1024
FLOP_PER_SAMPLE = 2.0 * (5.0 * math.log2(N_FFT) + 10.0)
INTER_BYTES_PER_SAMPLE = 2 * 2 * 8.0           # 2 segments per sample x (write + read) x 8 B


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:          # the numbers are still taken; the record says the query failed
        return {"name": None, "error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_scan.json"))
    args = ap.parse_args()
    import numpy as np
    import torch
    from habdec_b200 import api
    if not torch.cuda.is_available():
        raise SystemExit("bench_scan needs a CUDA device: nothing is measured without one")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    n_sms = torch.cuda.get_device_properties(0).multi_processor_count
    try:
        clk_mhz = float(info["max_sm_clock"].split()[0])
    except Exception:
        clk_mhz = float("nan")
    fp32_peak = n_sms * 128 * 2 * clk_mhz * 1e6

    # device copy bandwidth (read + write), 8 GB each way, best of 5
    a = torch.empty(8 << 30, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    best = 1e9
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); b.copy_(a); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    copy_gbs = 2 * a.numel() / (best * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()

    # ---- 1. standalone ------------------------------------------------------------------------------------------------
    gen = torch.Generator(device=dev); gen.manual_seed(4)
    caps = {api.IQ_CF32: (0.3 * torch.randn((1 << 29, 2), dtype=torch.float32, device=dev, generator=gen)),
            api.IQ_CS8: torch.randint(-128, 128, (1 << 31, 2), dtype=torch.int8, device=dev, generator=gen)}
    names = {api.IQ_CF32: "cf32", api.IQ_CS8: "cs8"}
    stream = torch.cuda.current_stream()
    scan = api.Scanner(N_FFT)
    scan.set_stream(stream.cuda_stream)

    def one_pass(fmt):
        cap = caps[fmt]
        n = cap.shape[0]
        scan.reset()
        for o in range(0, n, PUSH):
            scan.push_device(cap.data_ptr() + o * api.IQ_BYTES[fmt], min(PUSH, n - o), FS, fmt)
        return n

    for f in caps:                     # first use of every kernel and buffer
        one_pass(f)
    torch.cuda.synchronize()
    standalone = {names[f]: [] for f in caps}
    for rep in range(args.repeats):
        for f in (list(caps) if rep % 2 == 0 else list(caps)[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            n = one_pass(f)
            e1.record(stream)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            segs = scan.psd()[1]
            gsps = n / (ms * 1e-3) / 1e9
            t_fp32 = n * FLOP_PER_SAMPLE / fp32_peak
            t_hbm = n * api.IQ_BYTES[f] / (copy_gbs * 1e9)
            t_hbm_inter = n * (api.IQ_BYTES[f] + INTER_BYTES_PER_SAMPLE) / (copy_gbs * 1e9)
            standalone[names[f]].append({"ms": ms, "samples": n, "segments": segs, "gsps": gsps, "realtime_x_at_20msps": gsps * 1e9 / FS,
                                         "us_per_segment": ms * 1e3 / segs, "fp32_tflops": n * FLOP_PER_SAMPLE / (ms * 1e-3) / 1e12,
                                         "frac_fp32_bound": t_fp32 / (ms * 1e-3), "frac_hbm_bound_input": t_hbm / (ms * 1e-3),
                                         "frac_hbm_bound_if_intermediate_leaves_l2": t_hbm_inter / (ms * 1e-3)})
    # self-check: the CS8 pass and a cf32 pass over its dequantised first 2^24 samples agree bit for bit
    sub = caps[api.IQ_CS8][:1 << 24]
    deq = (sub.to(torch.float32) / 128.0).contiguous()
    s2 = api.Scanner(N_FFT)
    s2.set_stream(stream.cuda_stream)
    scan.reset()
    scan.push_device(sub.data_ptr(), sub.shape[0], FS, api.IQ_CS8)
    s2.push_device(deq.data_ptr(), sub.shape[0], FS)
    pa, pb = scan.psd(), s2.psd()
    check_equal = bool(pa[1] == pb[1] and np.array_equal(pa[0], pb[0]))
    del caps, sub, deq, s2
    torch.cuda.empty_cache()

    # ---- 2. beside the channeliser (configs[4]) -----------------------------------------------------------------------
    n_slices = 64
    gen.manual_seed(5)
    cap = 0.7 * torch.randn((n_slices * CHUNK, 2), dtype=torch.float32, device=dev, generator=gen)
    dec = api.BatchDecoder(N_CH, baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    dec.set_stream(stream.cuda_stream)
    for c in range(N_CH):
        dec.set_nco((c - N_CH / 2) * 15e3, c)
    scan.reset()
    done = [0]

    def step(with_scan):
        ptr = cap.data_ptr() + (done[0] % n_slices) * CHUNK * 8
        dec.pushWidebandDevice(ptr, CHUNK, FS)
        dec.process_async()
        if with_scan:
            scan.push_device(ptr, CHUNK, FS)
        done[0] += 1

    for i in range(3 * n_slices):
        step(i % 2 == 0)
        if (i + 1) % 16 == 0:
            dec.collect_ready(8)
    dec.collect()
    legs = {"channeliser": [], "channeliser_plus_scan": []}
    for rep in range(args.repeats):
        for with_scan in ((False, True) if rep % 2 == 0 else (True, False)):
            gc.collect(); gc.disable()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(args.steps):
                step(with_scan)
                if (k + 1) % 16 == 0:
                    dec.collect_ready(8)
            dec.collect()
            e1.record(stream)
            torch.cuda.synchronize()
            gc.enable()
            legs["channeliser_plus_scan" if with_scan else "channeliser"].append(e0.elapsed_time(e1) / args.steps)
    scan_segments = scan.psd()[1]

    def med(v): return float(np.median(v))
    summary = {k: {"gsps_median": med([x["gsps"] for x in v]), "gsps_spread": max(x["gsps"] for x in v) - min(x["gsps"] for x in v),
                   "us_per_segment_median": med([x["us_per_segment"] for x in v]),
                   "frac_fp32_bound_median": med([x["frac_fp32_bound"] for x in v]),
                   "frac_hbm_bound_input_median": med([x["frac_hbm_bound_input"] for x in v])} for k, v in standalone.items()}
    beside = {k: {"step_ms_median": med(v), "step_ms_spread": max(v) - min(v), "steps": v} for k, v in legs.items()}
    beside["added_fraction_median"] = beside["channeliser_plus_scan"]["step_ms_median"] / beside["channeliser"]["step_ms_median"] - 1.0
    beside["scan_segments_accumulated"] = scan_segments
    result = {"gpu": info, "n_fft": N_FFT, "push_samples": PUSH, "copy_gbs_read_plus_write": copy_gbs,
              "fp32_peak_tflops_computed": fp32_peak / 1e12, "flop_per_input_sample": FLOP_PER_SAMPLE,
              "standalone": standalone, "standalone_summary": summary, "cs8_equals_cf32_of_dequantised": check_equal,
              "beside_channeliser": beside,
              "note": "standalone: events around whole passes over a 4 GiB device capture (larger than L2) in 2^22-sample pushes; "
                      "beside: configs[4] step, 1024 channels, 65536-sample pushes, %d steps per leg, legs alternated over %d repeats"
                      % (args.steps, args.repeats)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"gpu": info, "standalone": summary, "beside": {k: v for k, v in beside.items() if k not in ("channeliser", "channeliser_plus_scan")} | {
        k: beside[k]["step_ms_median"] for k in ("channeliser", "channeliser_plus_scan")}, "check": check_equal}))
    if not check_equal:
        raise SystemExit("self-check failed: CS8 and cf32 of the dequantised samples differ")


if __name__ == "__main__":
    main()
