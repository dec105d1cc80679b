"""Cost of baud-rate estimation (hbd_set_baud_estimation) in the two benchmark geometries, estimation off against on:
  configs[3]  4096 channels at 2.048 MS/s, factor 256, device pushes from the HBM-resident ring of bench.py (300 baud 8N2,
              full-band SNR -15 dB; every step reads another 65 536-sample slice, the ring is far larger than L2);
  configs[4]  1024 NCO channels over a 20 MS/s device capture (512 MiB of noise, larger than L2), 65 536-sample wideband
              pushes.
Per geometry two handles on one stream, pipelined as in bench.py (collect_ready every 16 steps, lag 8), timed with CUDA
events over --steps steps and alternated off / on over --rounds rounds.  Also the wall time of one hbd_get_baud_estimates
(score kernel + copy, nothing in flight) on the handle with estimation on.  GPU name and power limit are read in the same
run.  Prints one JSON line; --out also writes it to a file.
usage: python tools/bench_baud.py [--steps 200] [--rounds 3] [--out profiles/r6_baud.json]"""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from habdec_b200 import api, synth

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=200)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--warmup", type=int, default=64)
ap.add_argument("--queries", type=int, default=20)
ap.add_argument("--out", default="")
a = ap.parse_args()
dev = torch.device("cuda", 0)
stream = torch.cuda.current_stream()
CHUNK = 65536


def measure(make, push):
    legs = {"off": make(), "on": make()}
    legs["on"].set_baud_estimation(True)
    pos = {k: 0 for k in legs}

    def step(k):
        push(legs[k], pos[k])
        pos[k] += 1
        legs[k].process_async()

    for k, d in legs.items():          # buffers sized, modules loaded, full frame cycles
        for i in range(a.warmup):
            step(k)
            if (i + 1) % 16 == 0:
                d.collect_ready(8)
        d.collect()
    ms = {k: [] for k in legs}
    for _ in range(a.rounds):
        for k, d in legs.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for i in range(a.steps):
                step(k)
                if (i + 1) % 16 == 0:
                    d.collect_ready(8)
            d.collect()
            e1.record(stream)
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / a.steps)
    q = []
    for _ in range(a.queries):
        t0 = time.perf_counter()
        est = legs["on"].baud_estimates()
        q.append((time.perf_counter() - t0) * 1e3)
    out = {k: {"ms_per_step_median": float(np.median(v)), "ms_per_step_all": [float(x) for x in v]} for k, v in ms.items()}
    out["step_ratio_on_over_off"] = out["on"]["ms_per_step_median"] / out["off"]["ms_per_step_median"]
    out["query_ms_median"] = float(np.median(q))
    out["query_ms_max"] = float(np.max(q))
    out["runs_per_channel_median"] = float(np.median(est["runs"]))
    out["nominal_300_share"] = float(np.mean(est["nominal"] == 300.0))
    for d in legs.values():
        d.close()
    return out


res = {}
# ---- configs[3]
N3, FS3 = 4096, 2.048e6
L = synth.ring_length(FS3, 300.0)
ring = synth.ring_iq_torch(0, N3, dev, FS3, 300.0, snr_db=-15.0)
torch.cuda.synchronize()


def make3():
    d = api.BatchDecoder(N3, baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    d.set_stream(stream.cuda_stream)
    d.set_raw_chars(False)
    return d


res["configs3"] = measure(make3, lambda d, i: d.pushSamplesDevice(ring.data_ptr() + (i % (L // CHUNK)) * CHUNK * 8, CHUNK, L, FS3))
res["configs3"]["workload"] = "%d channels, 2.048 MS/s cf32 device pushes of %d samples from the HBM ring, factor 256, 300 baud 8N2" % (N3, CHUNK)
del ring
torch.cuda.empty_cache()

# ---- configs[4]
N4, FS4, SLICES = 1024, 20e6, 64
cap = torch.randn((SLICES * CHUNK, 2), dtype=torch.float32, device=dev) * 0.7


def make4():
    d = api.BatchDecoder(N4, baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    d.set_stream(stream.cuda_stream)
    d.set_raw_chars(False)
    for c in range(N4):
        d.set_nco((c - N4 / 2) * 15e3, c)       # 15 kHz raster over the capture
    return d


res["configs4"] = measure(make4, lambda d, i: d.pushWidebandDevice(cap.data_ptr() + (i % SLICES) * CHUNK * 8, CHUNK, FS4))
res["configs4"]["workload"] = "wideband 20 MS/s device capture -> %d NCO channels, factor 256, %d-sample pushes" % (N4, CHUNK)

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
out = {"gpu": gpu, "steps": a.steps, "rounds": a.rounds, "pipeline": "collect_ready(8) every 16 steps", **res}
line = json.dumps(out)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
