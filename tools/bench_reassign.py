"""Cost of handing channels to new payloads (hbd_reset_channels) in the configs[4] geometry: 1024 NCO channels over a
20 MS/s HBM-resident capture, 65 536-sample device wideband pushes, pipelined as in tools/bench_wideband.py.  Two legs,
alternated over --repeats rounds on one handle each:
  steady  never resets;
  reset   first resets 64 channels spread over 16 consecutive calls (4 per call), so the channels sit on 16 FFT frame
          levels, then runs the same timed window.
Per leg: ms per step (median and spread over the rounds), host plan_call time and frame counters per call
(hbd_get_kernel_timing which 6), K4 launches per call, and the wall time of one hbd_reset_channels call (drain
included).  Prints one JSON line; --out also writes it to a file.
usage: python tools/bench_reassign.py [--steps 256] [--repeats 5] [--out profiles/r5_reassign.json]"""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from habdec_b200 import api

ap = argparse.ArgumentParser()
ap.add_argument("--channels", type=int, default=1024)
ap.add_argument("--steps", type=int, default=256)
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--chunk", type=int, default=65536)
ap.add_argument("--fs", type=float, default=20e6)
ap.add_argument("--out", default="")
a = ap.parse_args()
dev = torch.device("cuda", 0)
n_slices = 64
cap = torch.randn((n_slices * a.chunk, 2), dtype=torch.float32, device=dev) * 0.7   # 512 MiB: larger than L2
stream = torch.cuda.current_stream()


def make():
    d = api.BatchDecoder(a.channels, baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=256)
    d.set_stream(stream.cuda_stream)
    for c in range(a.channels):
        d.set_nco((c - a.channels / 2) * 15e3, c)                 # 15 kHz raster over the capture
    return d


legs = {"steady": make(), "reset": make()}
pos = {k: 0 for k in legs}


def step(name):
    d = legs[name]
    d.pushWidebandDevice(cap.data_ptr() + (pos[name] % n_slices) * a.chunk * 8, a.chunk, a.fs)
    pos[name] += 1
    d.process_async()


def launches_per_call(d, calls):
    # K1 + tail every call, K4 on the calls that complete a frame: K4 launches = total - 2 per call
    return (d.kernel_launches() - calls[0]) - 2 * calls[1]


for name in legs:       # warm-up: buffers sized, modules loaded, one full frame cycle
    for _ in range(32):
        step(name)
    legs[name].collect()
torch.cuda.synchronize()
rng = np.random.default_rng(5)
res = {k: {"ms_per_step": [], "plan_ms_per_call": [], "counters_per_call": [], "k4_per_call": [], "reset_call_ms": []} for k in legs}
for r in range(a.repeats):
    for name, d in legs.items():
        if name == "reset":    # 64 channels over 16 calls: 16 frame levels when the timed window starts
            chans = rng.choice(a.channels, 64, replace=False)
            for i in range(16):
                t0 = time.perf_counter()
                d.reset_channels(chans[4 * i:4 * i + 4])
                res[name]["reset_call_ms"].append((time.perf_counter() - t0) * 1e3)
                step(name)
                d.collect_ready(8)
            for _ in range(2):       # the first call after the last reset plans per channel
                step(name)
            d.collect()
        else:
            for _ in range(18):
                step(name)
            d.collect()
        torch.cuda.synchronize()
        d.set_kernel_timing(1)
        l0 = d.kernel_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(a.steps):
            step(name)
            if (i + 1) % 16 == 0:
                d.collect_ready(8)
        d.collect()
        e1.record(stream)
        torch.cuda.synchronize()
        plan_ms, counters = d.kernel_timing(6)
        k1_ms, k1_n = d.kernel_timing(0)
        res[name]["ms_per_step"].append(e0.elapsed_time(e1) / a.steps)
        res[name]["plan_ms_per_call"].append(plan_ms / a.steps)
        res[name]["counters_per_call"].append(counters / a.steps)
        res[name]["k4_per_call"].append(((d.kernel_launches() - l0) - 2 * a.steps) / a.steps)
        d.set_kernel_timing(0)

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
out = {"workload": "wideband %.0f MS/s -> %d NCO channels, dec=256, chunk %d, device pushes, pipelined (lag 8)" % (a.fs / 1e6, a.channels, a.chunk),
       "gpu": q, "steps": a.steps, "repeats": a.repeats}
for name, v in res.items():
    ms = np.array(v["ms_per_step"])
    leg = {"ms_per_step_median": float(np.median(ms)), "ms_per_step_min": float(ms.min()), "ms_per_step_max": float(ms.max()),
           "plan_ms_per_call": float(np.median(v["plan_ms_per_call"])), "frame_counters_per_call": float(np.median(v["counters_per_call"])),
           "k4_launches_per_call": float(np.median(v["k4_per_call"])), "ms_per_step_all": [float(x) for x in ms]}
    if v["reset_call_ms"]:
        rc = np.array(v["reset_call_ms"])
        leg.update(reset_call_ms_median=float(np.median(rc)), reset_call_ms_max=float(rc.max()))
    out[name] = leg
out["step_ratio_reset_over_steady"] = out["reset"]["ms_per_step_median"] / out["steady"]["ms_per_step_median"]
line = json.dumps(out)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
