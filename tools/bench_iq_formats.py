"""Integer IQ input at BASELINE configs[3] geometry (4096 channels x 65 536 samples per step, one GPU): cf32, CS16 and CS8
legs in one process, alternated, repeated.  Each format has its own HBM-resident ring (4096 x 1 638 400 samples: 54 / 27 /
13.5 GB, all larger than L2) fed through the zero-copy device push, so K1 streams 8, 4 or 2 bytes per sample.

Per leg: K1 ms per launch (CUDA events, hbd_set_kernel_timing(1)) and its share of its own HBM bound (8.125 / 4.125 / 2.125
B per sample against the device-to-device copy bandwidth measured here), the step (events around >= 40 steps with the
drains inside), and e2e from pinned host memory through hbd_push_iq_batch next to the H2D ceiling of the same buffers.
After the timed legs: every channel must have decoded its own ring sentence, and a slab of channels must equal the oracle
on the dequantised samples.  Writes profiles/r3_iq_formats.json (or --out).

    python tools/bench_iq_formats.py [--steps 40] [--repeats 3] [--out profiles/r3_iq_formats.json]
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FS, BAUD, CHUNK, N_CH, FACTOR, SCALE = 2.048e6, 300.0, 65536, 4096, 256, 1.0 / 32.0
K1_BYTES = {0: 8.125, 1: 4.125, 2: 2.125}          # per input sample: the input read + 8 B per 64 samples of stage-1 output
FIR_FLOP = 2.0 * 2.0 * 348 / 64                   # per input sample: T/M complex-by-real FMAs


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
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=6)
    ap.add_argument("--check-channels", type=int, default=32)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_iq_formats.json"))
    args = ap.parse_args()
    import numpy as np
    import torch
    from habdec_b200 import api, synth
    from oracle import pyoracle as po
    if not torch.cuda.is_available():
        raise SystemExit("bench_iq_formats needs a CUDA device: nothing is measured without one")
    dev = torch.device("cuda", 0)
    L = synth.ring_length(FS, BAUD)
    slices = L // CHUNK
    fmts = [api.IQ_CF32, api.IQ_CS16, api.IQ_CS8]
    names = {api.IQ_CF32: "cf32", api.IQ_CS16: "cs16", api.IQ_CS8: "cs8"}

    # rings: the cf32 ring holds the dequantised CS16 values, so all three legs decode the same signal
    rings = {api.IQ_CS16: torch.empty((N_CH, 2 * L), dtype=torch.int16, device=dev),
             api.IQ_CS8: torch.empty((N_CH, 2 * L), dtype=torch.int8, device=dev),
             api.IQ_CF32: torch.empty((N_CH, 2 * L), dtype=torch.float32, device=dev)}
    for c0 in range(0, N_CH, 512):
        r = torch.view_as_complex(synth.ring_iq_torch(c0, 512, dev, FS, BAUD, snr_db=-15.0))
        q16 = api.quantise(r, api.IQ_CS16, SCALE).reshape(512, -1)
        rings[api.IQ_CS16][c0:c0 + 512] = q16
        rings[api.IQ_CF32][c0:c0 + 512] = q16.to(torch.float32) / 32768.0
        rings[api.IQ_CS8][c0:c0 + 512] = api.quantise(r, api.IQ_CS8, SCALE).reshape(512, -1)
        del r, q16
    torch.cuda.synchronize()

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

    stream = torch.cuda.current_stream()
    decs, done = {}, {}
    for f in fmts:
        d = api.BatchDecoder(N_CH, baud=BAUD, rtty_bits=8, rtty_stops=2.0, dec_factor=FACTOR)
        d.set_stream(stream.cuda_stream)
        decs[f], done[f] = d, 0

    def step(f):
        ring = rings[f]
        d = decs[f]
        d.pushIQDevice(ring.data_ptr() + (done[f] % slices) * CHUNK * api.IQ_BYTES[f], f, CHUNK, L, FS)
        d.process_async()
        done[f] += 1

    for f in fmts:                     # one whole ring pass untimed: every kernel and host buffer has been through first use
        for i in range(slices + args.warmup):
            step(f)
            if (i + 1) % 8 == 0:
                decs[f].collect_ready(4)
        decs[f].collect()

    legs = {names[f]: [] for f in fmts}
    for rep in range(args.repeats):
        for f in (fmts if rep % 2 == 0 else fmts[::-1]):
            d = decs[f]
            d.set_kernel_timing(1)
            gc.collect(); gc.disable()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(args.steps):
                step(f)
                if (k + 1) % 8 == 0:
                    d.collect_ready(4)
            d.collect()
            e1.record(stream)
            torch.cuda.synchronize()
            gc.enable()
            k1_ms, k1_n = d.kernel_timing(0)
            d.set_kernel_timing(0)
            step_ms = e0.elapsed_time(e1) / args.steps
            k1 = k1_ms / max(k1_n, 1)
            samples = N_CH * CHUNK
            bound_ms = samples * K1_BYTES[f] / (copy_gbs * 1e9) * 1e3
            legs[names[f]].append({"k1_ms": k1, "k1_launches": k1_n, "k1_frac_of_hbm_bound": bound_ms / k1, "k1_hbm_bound_ms": bound_ms,
                                   "k1_fir_tflops": samples * FIR_FLOP / (k1 * 1e-3) / 1e12, "step_ms": step_ms,
                                   "gsps": samples / (step_ms * 1e-3) / 1e9})

    # e2e: pinned host buffers of each format -> hbd_push_iq_batch -> kernels; the H2D ceiling with the same buffers
    e2e = {}
    for f in fmts:
        host = [rings[f][:, i * 2 * CHUNK:(i + 1) * 2 * CHUNK].cpu().pin_memory() for i in range(3)]
        dst = torch.empty_like(host[0], device=dev)
        dst.copy_(host[0], non_blocking=True); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for h in host:
            dst.copy_(h, non_blocking=True)
        torch.cuda.synchronize()
        ceiling = sum(h.numel() * h.element_size() for h in host) / (time.perf_counter() - t0) / 1e9
        del dst
        d = api.BatchDecoder(N_CH, baud=BAUD, rtty_bits=8, rtty_stops=2.0, dec_factor=FACTOR)
        d.set_stream(stream.cuda_stream)

        def e2e_step(i):
            d._chk(d._lib.hbd_push_iq_batch(d._h, host[i % 3].data_ptr(), f, CHUNK, CHUNK, FS))
            d.process_async()
            d.collect_ready(1)
        e2e_step(0); d.collect()
        t0 = time.perf_counter()
        for i in range(args.e2e_steps):
            e2e_step(i + 1)
        d.collect(); torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        bytes_step = N_CH * CHUNK * api.IQ_BYTES[f]
        e2e[names[f]] = {"msps": N_CH * CHUNK * args.e2e_steps / dt / 1e6, "h2d_gbs": bytes_step * args.e2e_steps / dt / 1e9,
                         "h2d_gbs_ceiling": ceiling, "frac_of_h2d_ceiling": bytes_step * args.e2e_steps / dt / 1e9 / ceiling}
        d.close()
        del host

    # self-check: every channel's own CRC-valid ring sentence, and a slab against the oracle on the dequantised samples
    check = {}
    n_chk = args.check_channels
    cfg = po.make_config(baud=BAUD, rtty_bits=8, rtty_stops=2.0, dec_factor=FACTOR, record=False)
    kind = "ref" if po.available("ref") else "orc"
    for f in fmts:
        d = decs[f]
        chars = [d.poll_chars(c) for c in range(N_CH)]
        sents = [d.poll_sentences(c) for c in range(N_CH)]
        own = sum(1 for c in range(N_CH) if sents[c] and all(s == synth.ring_sentence(c).strip().lstrip("$").encode() for s in sents[c]))
        q = rings[f][:n_chk].cpu().numpy()
        iq = api.dequantise(q, f)
        ref_chars, ref_sents = po.run_ring(kind, cfg, iq, os.cpu_count() or 4, FS, CHUNK, 0, done[f])
        slab_ok = all(chars[c] == ref_chars[c] and sents[c] == ref_sents[c] for c in range(n_chk))
        check[names[f]] = {"channels_with_own_sentence": own, "channels": N_CH, "oracle": kind, "oracle_slab_channels": n_chk,
                           "oracle_slab_equal": slab_ok, "steps": done[f]}

    def summary(name):
        v = legs[name]
        k1 = [x["k1_ms"] for x in v]
        st = [x["step_ms"] for x in v]
        return {"k1_ms_median": float(np.median(k1)), "k1_ms_spread": float(max(k1) - min(k1)), "step_ms_median": float(np.median(st)),
                "step_ms_spread": float(max(st) - min(st)), "k1_frac_of_hbm_bound_median": float(np.median([x["k1_frac_of_hbm_bound"] for x in v])),
                "gsps_median": float(np.median([x["gsps"] for x in v]))}
    summ = {n: summary(n) for n in legs}
    result = {"gpu": gpu_info(), "geometry": {"channels": N_CH, "chunk": CHUNK, "fs": FS, "factor": FACTOR, "ring_samples_per_channel": L},
              "copy_gbs_read_plus_write": copy_gbs, "k1_bytes_per_sample": {names[f]: K1_BYTES[f] for f in fmts},
              "fir_flop_per_sample": FIR_FLOP, "legs": legs, "summary": summ,
              "k1_ratio_cs16_over_cf32": summ["cs16"]["k1_ms_median"] / summ["cf32"]["k1_ms_median"],
              "k1_ratio_cs8_over_cf32": summ["cs8"]["k1_ms_median"] / summ["cf32"]["k1_ms_median"],
              "step_ratio_cs16_over_cf32": summ["cs16"]["step_ms_median"] / summ["cf32"]["step_ms_median"],
              "e2e": e2e, "self_check": check,
              "note": "device pushes from HBM-resident rings larger than L2; K1 from CUDA events around every launch; step = events around "
                      "%d steps per leg with drains inside, legs alternated over %d repeats" % (args.steps, args.repeats)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"summary": summ, "e2e": e2e, "check": check, "gpu": result["gpu"],
                      "k1_ratio_cs16_over_cf32": result["k1_ratio_cs16_over_cf32"]}))
    ok = all(c["channels_with_own_sentence"] == N_CH and c["oracle_slab_equal"] for c in check.values())
    if not ok:
        raise SystemExit("self-check failed: %r" % check)


if __name__ == "__main__":
    main()
