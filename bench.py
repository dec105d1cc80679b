#!/usr/bin/env python
"""bench.py -- aggregate IQ MSamples/s decoded (BASELINE.json metric) on N B200s of one node.

Workload (BASELINE.json configs[3]): independent RTTY channels, fs 2.048 MS/s, 300 baud 8N2, 425 Hz shift, dec=8
(factor 256), low-pass 1500 Hz, block-partitioned over the ranks.  There is no collective on the signal path; the
decoded characters / sentences / AFC scalars of every channel are gathered to rank 0 as fixed-size records over NCCL
(hbd_gather_results, csrc/dist.cu) INSIDE the timed region, once per drain.  One "step" = one Decoder::process() over one
65 536-sample chunk of every channel.  Inputs are synthetic (habdec_b200/synth.py ring workload: periodic
continuous-phase FSK + AWGN, one CRC-valid 21-character sentence per 25 chunks), resident in HBM for `value`, in pinned
host memory for `e2e`.

The run proves its own metric ("chars bit-exact"): after the timed region every local channel's characters and sentences
are compared with the reference Decoder (oracle/_ref, one Decoder per channel on the host threads) over exactly the chunks
the GPU decoded; a mismatch makes the run fail.

Legs of one invocation (all on the same JSON line):
  value / roofline / e2e   weak scaling, 4096 channels per GPU (configs[3] as the per-GPU shard)
  strong                   configs[3] as written: 4096 channels IN TOTAL over the N GPUs (N = 1: the weak leg itself)
  wideband                 configs[4]: one 20 MS/s capture -> 1024 NCO channels (N = 1 only; --no-wideband skips it)

  python bench.py --gpus 1 --steps 20 --warmup 5            # our arm
  python bench.py --impl reference --steps 3 --warmup 1     # the reference's CPU Decoder on the host cores
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: importing the package must not write __pycache__ into it

import numpy as np  # noqa: E402

FS = 2.048e6
BAUD = 300.0
FACTOR = 256
TOTAL_CHANNELS = 4096
SNR_DB = -15.0
ALGO_BYTES_PER_SAMPLE_K1 = 8.0 + 8.0 / 64.0   # cf32 read + stage-1 output write (DESIGN.md section 4)
ALGO_BYTES_PER_SAMPLE_STEP = 8.0 + 12.0 / 256.0  # SURVEY 8(d): cf32 read + (demod 4 + decimated IQ 8) / 256
# DRAM bytes per input sample that K1 really moved in the ncu --set full capture of this exact workload
# (profiles/r2_k1_ncu_full_raw.csv: dram__bytes_read.sum 2.172891 GB + dram__bytes_write.sum 0.009870 GB per 2^28 samples;
# round 1, before the L2 evict-first hint on the input stream: 2.170465 + 0.046897 GB)
NCU_TRAFFIC_BYTES_PER_SAMPLE_K1 = (2.172891e9 + 0.009870e9) / 268435456.0
FP32_PEAK_TFLOPS = 73.8                        # measured with tools/micro/ffma2_bench.cu on this pool's B200 (DESIGN.md section 4)
METRIC = "aggregate IQ MSamples/s decoded (chars bit-exact)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--channels", type=int, default=None, help="total channels of the weak leg (default: 4096 per GPU)")
    ap.add_argument("--chunk", type=int, default=65536, help="complex samples per channel per step")
    ap.add_argument("--e2e-steps", type=int, default=6)
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="target duration of the cpu_baseline leg")
    ap.add_argument("--collect-every", type=int, default=4, help="drain finished calls every this many steps")
    ap.add_argument("--gather-every", type=int, default=0, help="gather the result records to rank 0 every this many steps; 0: once per batch, after the last step")
    ap.add_argument("--collect-lag", type=int, default=3, help="calls left in flight by the periodic drain")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="diagnostic: skip the all-channel comparison with the reference Decoder")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-wideband", action="store_true")
    ap.add_argument("--no-kernel-timing", action="store_true", help="diagnostic: no CUDA events around K1 (no roofline numbers)")
    ap.add_argument("--pipeline-diagnostics", action="store_true", help="also time the rest of the step (two more event records per call): rest_of_step_ms, pipeline_gaps")
    ap.add_argument("--no-pin", action="store_true", help="diagnostic: leave the CPU affinity alone")
    ap.add_argument("--ref-passes", type=int, default=8, help="reference arm: ring passes per host thread per step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the weak leg, write what its caller holds (rank 0's channels) as DIR/<name>.npy, float32/float64, "
                         "under 64 MB; the inputs are seeded, so two builds can be compared array for array")
    a = ap.parse_args()
    if a.channels is None:
        world = int(os.environ.get("WORLD_SIZE", "1"))   # ranks actually launched (torchrun); --gpus is informational
        a.channels = TOTAL_CHANNELS * max(world, 1)
    return a


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons sampled (NVML, every few ms) while the timed region runs."""

    def __init__(self, index):
        self.index, self.rows, self._stop, self.th = index, [], False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.mx = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
            return
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def _run(self):
        nv = self.nv
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        rs, k = 0, 0
        while not self._stop:
            try:
                clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                if k % 3 == 0:          # NVML queries can take tens of ms on a busy box: the clock every time, the reasons every third
                    rs = reasons(self.h)
                k += 1
                self.rows.append((clk, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self):
        self._stop = True
        if self.th:
            self.th.join(timeout=1.0)
        if not getattr(self, "nv", None) or not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        nv = self.nv
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8), "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        reasons = sorted({name for _, rs in self.rows for name, b in bits.items() if rs & b})
        return {"sm_mhz": float(np.median([c for c, _ in self.rows])), "sm_max_mhz": float(self.mx), "reasons": reasons, "samples": len(self.rows)}


def workload_config(args, world):
    return {"workload": "BASELINE configs[3]: %d RTTY channels per GPU (%d in total, weak scaling), 2.048 MS/s cf32, 300 baud 8N2, 425 Hz shift, "
                        "dec=8 (factor 256), lowpass 1500 Hz, chunk %d samples/channel/step" % (args.channels // world, args.channels, args.chunk),
            "channels_total": args.channels, "channels_per_gpu": args.channels // world, "chunk": args.chunk,
            "snr_db_fullband": SNR_DB, "l2_policy": "inputs larger than L2: every step reads a different %.2f GiB slice of a ring resident in HBM"
            % (args.channels // world * args.chunk * 8 / 2**30), "parallelism": "channels block-partitioned, %d rank(s)" % world}


# ---------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CPU Decoder (oracle/_ref when it was built, else the restatement) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from habdec_b200 import synth
    from oracle import pyoracle as po
    kind = "ref" if po.available("ref") else "orc"
    cores = os.cpu_count() or 1
    cfg = po.make_config(baud=BAUD, rtty_bits=8, rtty_stops=2.0, lowpass_bw=1500.0, lowpass_trans=0.025, dec_factor=FACTOR, record=False)
    L = synth.ring_length(FS, BAUD)
    iq = np.stack([synth.ring_iq_numpy(c, FS, BAUD, snr_db=SNR_DB) for c in range(cores)])
    # a step = every host thread decodes `ref_passes` ring passes (L samples each) of its own channel, pushed in
    # `chunk` pieces exactly like DECODER_THREAD does (code/websocketServer/main.cpp:235-245)
    P = max(1, args.ref_passes)
    if args.warmup > 0:
        po.bench(kind, cfg, iq, cores, FS, chunk=args.chunk, reps=P * args.warmup)
    t0 = time.time()
    secs, chars = po.bench(kind, cfg, iq, cores, FS, chunk=args.chunk, reps=P * args.steps)
    wall = time.time() - t0
    samples = float(cores) * L * P * args.steps
    value = samples / secs / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "MSamples/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": secs * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, max(int(os.environ.get("WORLD_SIZE", "1")), 1)),
            "cpu_baseline": {"value": value, "unit": "MSamples/s", "cores": cores, "kind": "reference" if kind == "ref" else "port",
                             "sample": "%d host threads x %d steps x %d ring passes of %d samples each (one Decoder per thread), wall %.1f s, %d chars decoded"
                             % (cores, args.steps, P, L, wall, chars)},
            "e2e": {"value": value, "unit": "MSamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------
class Dist:
    """torch.distributed for the harness plumbing (barriers, max over ranks, handing out the NCCL id)."""

    def __init__(self):
        import torch
        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            import torch.distributed as dist
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def all_values(self, x: float) -> list:
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [float(x)]
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(v.item()) for v in out]

    def sum_int(self, x: int) -> int:
        t = self.torch.tensor([x], dtype=self.torch.int64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t)
        return int(t.item())

    def share_bytes(self, b: bytes | None, n: int) -> bytes:
        t = self.torch.zeros(n, dtype=self.torch.uint8, device=self.dev)
        if self.rank == 0:
            t.copy_(self.torch.frombuffer(bytearray(b), dtype=self.torch.uint8))
        if self.world > 1:
            self.dist.broadcast(t, src=0)
        return bytes(t.cpu().numpy())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def pin_cores(D: Dist):
    """One block of host cores per rank: the issuing thread, the drain and the parity threads of a rank stay off the
    other ranks' cores (the N = 8 straggler of round 1 was a host thread, not a kernel)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = max(1, len(cores) // D.world)
        mine = cores[D.local_rank * per:(D.local_rank + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return mine
    except Exception:
        return None


def decode_leg(D: Dist, args, n_local, ch0, n_total, steps, warmup, timing=True, sample_clocks=True):
    """One weak- or strong-scaling run: ring in HBM -> preroll + warmup (untimed) -> `steps` timed steps with periodic
    drains and NCCL gathers -> final drain + gather.  Returns a dict of measurements plus what the parity check needs."""
    torch = D.torch
    from habdec_b200 import api, synth
    L = synth.ring_length(FS, BAUD)
    assert L % args.chunk == 0, "chunk must divide the ring length %d" % L
    slices = L // args.chunk
    ring = synth.ring_iq_torch(ch0, n_local, D.dev, FS, BAUD, snr_db=SNR_DB)          # [n_local, L, 2] float32, HBM resident
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    dec = api.BatchDecoder(n_local, device=D.local_rank, baud=BAUD, rtty_bits=8, rtty_stops=2.0, lowpass_bw=1500.0, lowpass_trans=0.025,
                           dec_factor=FACTOR)
    dec.set_stream(stream.cuda_stream)
    dec.set_raw_chars(False)            # nobody polls the unfiltered characters here (the reference keeps none either)
    uid = D.share_bytes(api.dist_unique_id() if (D.rank == 0 and D.world > 1) else None, 128) if D.world > 1 else None
    dec.dist_init(D.rank, D.world, uid)                     # NCCL communicator owned by the library (csrc/dist.cu)
    sink = api.ResultSink(n_total)                          # rank 0: every channel; other ranks: a mirror of their own block
    base_ptr = ring.data_ptr()
    # the stream starts at the beginning of the ring and runs one whole ring pass before anything is timed (every kernel of the
    # path -- the FFT/AFC kernel runs once per 16 calls -- and every per-channel host buffer has then been through its first
    # use); the rest of the untimed part is sized so that a sentence (extracted by the call that sees ring chunk 0 again) falls
    # into the middle of a 20-step timed region: preroll + warmup = 15 (mod 25)
    preroll = slices + (15 - warmup) % slices
    n_done = 0

    def step():
        nonlocal n_done
        dec.pushSamplesDevice(base_ptr + (n_done % slices) * args.chunk * 8, args.chunk, L, FS)
        dec.process_async()
        n_done += 1

    for _ in range(preroll + warmup):
        step()
        if n_done % args.collect_every == 0:
            dec.collect_ready(args.collect_lag)
    dec.collect()
    dec.gather_results(sink)
    launches0 = dec.kernel_launches()
    dec.set_kernel_timing((2 if args.pipeline_diagnostics else 1) if timing else 0)
    sampler = ClockSampler(D.local_rank) if sample_clocks else None
    if sampler:
        sampler.start()                  # every rank watches its own GPU (a throttled GPU shows up as a slow rank)
    gc.collect()
    gc.disable()                         # no collector pause of the Python harness inside a 2..8 ms timed region
    D.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    t_issue = t_drain = 0.0
    issue_max = drain_max = 0.0
    gathers = 0
    for k in range(steps):
        t_h = time.perf_counter()
        step()
        dt_h = time.perf_counter() - t_h
        t_issue += dt_h
        issue_max = max(issue_max, dt_h)
        if (k + 1) % args.collect_every == 0:
            t_h = time.perf_counter()
            dec.collect_ready(args.collect_lag)   # drain finished calls; the newest few stay in flight so the GPU never idles
            if args.gather_every and (k + 1) % args.gather_every == 0:
                dec.gather_results(sink)          # records of every channel -> rank 0 (NCCL send/recv)
                gathers += 1
            dt_h = time.perf_counter() - t_h
            t_drain += dt_h
            drain_max = max(drain_max, dt_h)
    t_fc = time.perf_counter()
    dec.collect()                       # results drained (D2H + sentence layer) inside the timed region
    t_fg = time.perf_counter()
    dec.gather_results(sink)
    gathers += 1
    final_ms = (time.perf_counter() - t_fc) * 1e3
    final_gather_ms = (time.perf_counter() - t_fg) * 1e3
    ev1.record(stream)
    gc.enable()
    D.barrier()
    clocks = sampler.stop() if sampler else {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    ms = ev0.elapsed_time(ev1)
    k1_ms, k1_cnt = dec.kernel_timing(0) if timing else (0.0, 0)
    rest_ms, rest_cnt = dec.kernel_timing(1) if timing else (0.0, 0)
    gaps = {}
    if timing and args.pipeline_diagnostics:
        for name, w in (("k1_end_to_next_k1_start_ms", 2), ("k1_end_to_tail_start_ms", 3), ("tail_end_to_k1_plus2_start_ms", 4)):
            g_ms, g_cnt = dec.kernel_timing(w)
            gaps[name] = g_ms / g_cnt if g_cnt else None
    replay_ms, replay_calls = dec.kernel_timing(5) if timing else (0.0, 0)
    dec.set_kernel_timing(False)
    launches = dec.kernel_launches() - launches0
    # characters that did not fit the last records (more than 256 pending in one channel): flush them, untimed
    for _ in range(8):
        if not any(dec.poll_chars(c) for c in (0, n_local // 2, n_local - 1)):
            break
        dec.gather_results(sink)
    # the sink hands each stream out once: take this rank's channels here for the parity check and --dump-outputs
    got = [(sink.poll_chars(g), sink.poll_sentences(g)) for g in range(ch0, ch0 + n_local)]
    per_rank_diag = {"k1_avg_ms": D.all_values(k1_ms / max(k1_cnt, 1)), "host_replay_ms_total": D.all_values(replay_ms),
                     "issue_max_ms": D.all_values(issue_max * 1e3), "drain_max_ms": D.all_values(drain_max * 1e3), "final_ms": D.all_values(final_ms), "final_gather_ms": D.all_values(final_gather_ms),
                     "sm_mhz": D.all_values(float(clocks["sm_mhz"] or 0)), "throttle_reasons": D.all_values(float(len(clocks["reasons"])))}
    per_rank_ms = D.all_values(ms)
    per_rank_issue = D.all_values(t_issue * 1e3 / max(steps, 1))
    per_rank_drain = D.all_values((t_drain * 1e3 + final_ms) / max(steps, 1))
    return {"dec": dec, "sink": sink, "got": got, "ring": ring, "ms": ms, "ms_max": max(per_rank_ms), "per_rank_ms": per_rank_ms,
            "per_rank_issue_ms": per_rank_issue, "per_rank_drain_ms": per_rank_drain, "per_rank_diag": per_rank_diag, "k1_ms": k1_ms, "k1_cnt": k1_cnt,
            "rest_ms": rest_ms, "rest_cnt": rest_cnt, "gaps": gaps, "launches": launches, "clocks": clocks, "final_ms": final_ms,
            "chunks_decoded": n_done, "preroll": preroll, "gathers": gathers, "L": L}


def parity_check(D: Dist, args, leg, n_local, ch0):
    """Every local channel against the reference Decoder over exactly the chunks this leg decoded (outside all timing)."""
    from oracle import pyoracle as po
    kind = "ref" if po.available("ref") else "orc"
    cfg = po.make_config(baud=BAUD, rtty_bits=8, rtty_stops=2.0, lowpass_bw=1500.0, lowpass_trans=0.025, dec_factor=FACTOR, record=False)
    try:
        threads = len(os.sched_getaffinity(0))
    except Exception:
        threads = os.cpu_count() or 1
    ring, L = leg["ring"], leg["L"]
    torch = D.torch
    t0 = time.time()
    bad, n_chars, n_sent, sent_min = [], 0, 0, None
    slab = 128
    # the ring goes back to the host slab by slab through two pinned buffers; the copy of the next slab runs while the
    # host threads decode the current one
    bufs = [torch.empty((slab, L, 2), dtype=torch.float32, pin_memory=True) for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    events = [None, None]

    def fetch(i):
        c0 = i * slab
        c1 = min(n_local, c0 + slab)
        with torch.cuda.stream(copy_stream):
            bufs[i % 2][:c1 - c0].copy_(ring[c0:c1], non_blocking=True)
            events[i % 2] = torch.cuda.Event()
            events[i % 2].record(copy_stream)

    n_slabs = (n_local + slab - 1) // slab
    fetch(0)
    for i in range(n_slabs):
        c0 = i * slab
        c1 = min(n_local, c0 + slab)
        events[i % 2].synchronize()
        if i + 1 < n_slabs:
            fetch(i + 1)
        iq = bufs[i % 2][:c1 - c0].numpy().view(np.complex64).reshape(c1 - c0, L)
        ref_chars, ref_sents = po.run_ring(kind, cfg, iq, threads, FS, args.chunk, 0, leg["chunks_decoded"])
        for k in range(c1 - c0):
            g = ch0 + c0 + k
            got_c, got_s = leg["got"][c0 + k]
            n_chars += len(ref_chars[k]); n_sent += len(ref_sents[k])
            sent_min = len(got_s) if sent_min is None else min(sent_min, len(got_s))
            if got_c != ref_chars[k] or got_s != ref_sents[k]:
                bad.append(g)
    del bufs
    checked = D.sum_int(n_local)
    mism = D.sum_int(len(bad))
    smin = int(min(D.all_values(float(sent_min or 0))))
    return {"channels_checked": checked, "mismatches": mism, "first_bad": bad[:4], "oracle": "reference" if kind == "ref" else "port",
            "chunks_per_channel": leg["chunks_decoded"], "chars_compared": D.sum_int(n_chars), "sentences_compared": D.sum_int(n_sent),
            "sentences_min": smin, "seconds": round(time.time() - t0, 1), "host_threads_per_rank": threads}


DUMP_TAIL = 512                 # newest bytes kept of each channel's character and sentence streams (a step adds about one)
DUMP_POWER_CHANNELS = 256       # power spectra are fft_n floats per channel: a fixed sample of channels


def dump_outputs(out_dir, leg, n_local, ch0):
    """What the caller of the weak leg holds after its last timed step, for comparing two builds output for output:
    the newest characters and sentences gathered per channel, the newest record's scalars (frequency correction, shift,
    noise floor, noise variance, left and right peak), the last step's demodulated block and the current power spectrum.
    Rows are padded with NaN; characters are byte values.  Channels (local numbers in channels.npy) are a fixed, seeded
    sample where all of them would exceed 64 MB."""
    dec, sink = leg["dec"], leg["sink"]

    def rows(items):
        a = np.full((len(items), max([len(x) for x in items] + [1])), np.nan, dtype=np.float32)
        for i, x in enumerate(items):
            a[i, :len(x)] = x
        return a

    rng = np.random.default_rng(20240601)
    demod_w = max(len(dec.getDemodulated(0)), 1)
    per_channel = 4 * (2 * DUMP_TAIL + demod_w) + 8 * 7
    n = min(n_local, (48 << 20) // per_channel)          # + at most 16 MB of power spectra
    chans = np.arange(n_local) if n == n_local else np.sort(rng.choice(n_local, n, replace=False))
    tail = lambda b: np.frombuffer(b[-DUMP_TAIL:], dtype=np.uint8)
    stats = [sink.stats(ch0 + int(c)) for c in chans]
    pchans = chans if n <= DUMP_POWER_CHANNELS else np.sort(rng.choice(chans, DUMP_POWER_CHANNELS, replace=False))
    out = {"channels": chans.astype(np.float64),
           "chars": rows([tail(leg["got"][c][0]) for c in chans]),
           "sentences": rows([tail(b"".join(s + b"\n" for s in leg["got"][c][1])) for c in chans]),
           "stats": np.stack([s if s is not None else np.full(6, np.nan) for s in stats]).astype(np.float64),
           "demodulated": rows([dec.getDemodulated(int(c)) for c in chans]),
           "power_spectrum": rows([dec.getPowerSpectrum(int(c)) for c in pchans]),
           "power_spectrum_channels": pchans.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_e2e(D: Dist, args, ring, C):
    """Same metric through the C ABI with HOST buffers (H2D of every step's input + D2H of results in the timed region)."""
    torch = D.torch
    from habdec_b200 import api
    stream = torch.cuda.current_stream()
    n_host = 3
    host = [torch.empty((C, args.chunk, 2), dtype=torch.float32, pin_memory=True) for _ in range(n_host)]
    for i in range(n_host):
        host[i].copy_(ring[:, i * args.chunk:(i + 1) * args.chunk, :])
    torch.cuda.synchronize()
    # the ceiling: the same buffers copied with nothing else going on, all ranks at once
    dst = torch.empty((C, args.chunk, 2), dtype=torch.float32, device=D.dev)
    dst.copy_(host[0], non_blocking=True)
    D.barrier()
    t0 = time.perf_counter()
    for i in range(n_host):
        dst.copy_(host[i], non_blocking=True)
    torch.cuda.synchronize()
    h2d_s = max(D.all_values(time.perf_counter() - t0))
    del dst
    dec2 = api.BatchDecoder(C, device=D.local_rank, baud=BAUD, rtty_bits=8, rtty_stops=2.0, dec_factor=FACTOR)
    dec2.set_stream(stream.cuda_stream)

    def e2e_step(i):
        # host buffer -> hbd_push_samples_batch (H2D inside, the caller owns the buffer again on return) -> kernels;
        # the results of the previous step are read back (D2H + sentence layer) while this step's kernels run
        h = host[i % n_host]
        dec2._chk(dec2._lib.hbd_push_samples_batch(dec2._h, h.data_ptr(), args.chunk, args.chunk, FS))
        dec2.process_async()
        dec2.collect_ready(1)
    e2e_step(0)
    dec2.collect()
    D.barrier()
    t0 = time.perf_counter()
    for i in range(args.e2e_steps):
        e2e_step(i + 1)
    dec2.collect()                  # the last step's results
    torch.cuda.synchronize()
    dt = max(D.all_values(time.perf_counter() - t0))
    d2h = sum(len(dec2.poll_raw_chars(c)) for c in range(C)) * 8 / max(args.e2e_steps + 1, 1) + 32
    bytes_step = C * args.chunk * 8
    ceiling = D.world * bytes_step * n_host / h2d_s / 1e9
    out = {"value": float(C * D.world) * args.chunk * args.e2e_steps / dt / 1e6, "unit": "MSamples/s",
           "h2d_bytes_per_step": int(bytes_step), "d2h_bytes_per_step": int(d2h), "steps": args.e2e_steps,
           "h2d_gbs_achieved": D.world * bytes_step * args.e2e_steps / dt / 1e9, "h2d_gbs_ceiling": ceiling,
           "frac_of_h2d_ceiling": (D.world * bytes_step * args.e2e_steps / dt / 1e9) / ceiling,
           "note": "hbd_push_samples_batch from pinned host memory + hbd_process_async + hbd_collect_ready per step, wall clock, max over ranks; "
                   "PCIe bound: h2d_gbs_ceiling is the same pinned buffers copied by all %d rank(s) at once with nothing else running" % D.world}
    dec2.close()
    return out


def run_wideband(D: Dist, args):
    """BASELINE configs[4] (N = 1): one 20 MS/s capture -> 1024 frequency-offset channels through the NCO fused into K1."""
    torch = D.torch
    from habdec_b200 import api
    fs, n_ch, chunk, steps = 20e6, 1024, 65536, 40
    n_slices = 64
    gen = torch.Generator(device=D.dev)
    gen.manual_seed(2024)
    cap = torch.randn((n_slices * chunk, 2), dtype=torch.float32, device=D.dev, generator=gen) * 0.7
    dec = api.BatchDecoder(n_ch, device=D.local_rank, baud=300.0, rtty_bits=8, rtty_stops=2.0, dec_factor=FACTOR)
    stream = torch.cuda.current_stream()
    dec.set_stream(stream.cuda_stream)
    dec.set_raw_chars(False)
    for c in range(n_ch):
        dec.set_nco((c - n_ch / 2) * 15e3, c)                    # 15 kHz raster over the capture
    done = 0

    def step():
        nonlocal done
        dec.pushWidebandDevice(cap.data_ptr() + (done % n_slices) * chunk * 8, chunk, fs)
        dec.process_async()
        done += 1
    for _ in range(5):
        step()
    dec.collect()
    torch.cuda.synchronize()
    dec.set_kernel_timing(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(steps):
        step()
        if (k + 1) % 8 == 0:
            dec.collect_ready(4)
    dec.collect()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    k1_ms, k1_n = dec.kernel_timing(0)
    dec.set_kernel_timing(False)
    k1 = k1_ms / max(k1_n, 1)
    flops = (4.0 * 348 / 64 + 10.0) * n_ch * chunk             # FIR 21.75 + complex mix 10 flop per channel-sample (DESIGN.md section 4)
    dec.close()
    return {"workload": "BASELINE configs[4]: one 20 MS/s capture -> %d NCO channels (15 kHz raster), dec=8, chunk %d; noise capture, "
                        "parity of this path: tests/test_gpu_nco.py" % (n_ch, chunk),
            "channel_MSamples_per_s": n_ch * chunk / (ms * 1e-3) / 1e6, "realtime_factor": chunk / (ms * 1e-3) / fs, "ms_per_step": ms,
            "k1_nco_avg_ms": k1, "k1_nco_tflops": flops / (k1 * 1e-3) / 1e12 if k1 else None,
            "fp32_frac": flops / (k1 * 1e-3) / 1e12 / FP32_PEAK_TFLOPS if k1 else None, "fp32_peak_tflops": FP32_PEAK_TFLOPS, "steps": steps}


def run_ours(args):
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: habdec_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    D = Dist()
    cores = None if args.no_pin else pin_cores(D)
    from habdec_b200 import synth
    world, rank = D.world, D.rank
    assert args.channels % world == 0
    C = args.channels // world
    ch0 = rank * C

    # ---- weak leg: the headline ------------------------------------------------------------------------
    leg = decode_leg(D, args, C, ch0, args.channels, args.steps, args.warmup, timing=not args.no_kernel_timing)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, leg, C, ch0)
    ms_max = leg["ms_max"]
    total_samples = float(args.channels) * args.chunk * args.steps
    value = total_samples / (ms_max * 1e-3) / 1e6
    parity = None if args.no_parity else parity_check(D, args, leg, C, ch0)
    totals = leg["sink"].totals() if rank == 0 else None
    result_hash = "%016x" % leg["sink"].hash() if rank == 0 else None

    e2e = None if args.no_e2e else run_e2e(D, args, leg["ring"], C)
    leg["dec"].dist_finalize()
    leg["dec"].close()
    ring_bytes = leg["ring"].numel() * 4
    del leg["ring"], leg["dec"]
    torch.cuda.empty_cache()

    # ---- strong leg: configs[3] as written, 4096 channels in total --------------------------------------
    strong = None
    if not args.no_strong:
        if world == 1 and args.channels == TOTAL_CHANNELS:
            strong = {"channels_total": TOTAL_CHANNELS, "channels_per_gpu": C, "value": value, "ms_per_step": ms_max / args.steps,
                      "speedup_vs_one_gpu": 1.0, "result_hash": result_hash, "parity": parity, "note": "N = 1: the weak leg is configs[3] as written"}
        elif TOTAL_CHANNELS % (world * 32) == 0:
            Cs = TOTAL_CHANNELS // world
            # no NVML polling here: the clocks line of the JSON is the weak leg's, and this leg's timed region is only 2..4 ms
            sleg = decode_leg(D, args, Cs, rank * Cs, TOTAL_CHANNELS, args.steps, args.warmup, timing=False, sample_clocks=False)
            s_value = float(TOTAL_CHANNELS) * args.chunk * args.steps / (sleg["ms_max"] * 1e-3) / 1e6
            s_par = None if args.no_parity else parity_check(D, args, sleg, Cs, rank * Cs)
            strong = {"channels_total": TOTAL_CHANNELS, "channels_per_gpu": Cs, "value": s_value, "ms_per_step": sleg["ms_max"] / args.steps,
                      # one GPU's throughput on the whole of configs[3] is the per-GPU rate of the weak leg (4096 channels per GPU, same run)
                      "speedup_vs_one_gpu": s_value / (value / world), "efficiency_vs_n1": s_value / (value / world) / world,
                      "per_rank_ms": sleg["per_rank_ms"], "per_rank_host_issue_ms_per_step": sleg["per_rank_issue_ms"],
                      "per_rank_host_drain_ms_per_step": sleg["per_rank_drain_ms"], "gathers_in_timed_region": sleg["gathers"],
                      "result_hash": ("%016x" % sleg["sink"].hash()) if rank == 0 else None, "parity": s_par,
                      "note": "result_hash covers every channel's character and sentence streams as gathered on rank 0: identical for N = 1, 2, 4, 8"}
            sleg["dec"].dist_finalize()
            sleg["dec"].close()
            del sleg
            torch.cuda.empty_cache()

    wideband = None
    if world == 1 and not args.no_wideband:
        wideband = run_wideband(D, args)

    if rank != 0:
        D.close()
        if parity and parity["mismatches"]:
            sys.exit(3)
        return

    peak, peak_src = load_peaks()
    k1_cnt, k1_ms = leg["k1_cnt"], leg["k1_ms"]
    # K1 is launched once per step: algorithmic bytes of one launch = the step's samples x 8.125 B
    k1_bytes = ALGO_BYTES_PER_SAMPLE_K1 * C * args.chunk * args.steps / max(k1_cnt, 1)
    k1_avg_ms = k1_ms / max(k1_cnt, 1)
    achieved = k1_bytes / (k1_avg_ms * 1e-3) / 1e9 if k1_cnt else None
    step_gbs = ALGO_BYTES_PER_SAMPLE_STEP * C * args.chunk / (ms_max / args.steps * 1e-3) / 1e9
    line = {"metric": METRIC, "value": value, "unit": "MSamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": dict(workload_config(args, world), preroll_steps=leg["preroll"],
                                                  ring="one 21-character CRC-valid sentence per 25 chunks and channel; the stream starts at the ring start, "
                                                       "%d untimed steps (one ring pass + alignment + warmup) precede the timed region" % (leg["preroll"] + args.warmup),
                                                  ring_bytes_per_gpu=ring_bytes, host_cores_of_rank0=cores),
            "roofline": {"bound": "hbm", "kernel": "decim1_kernel<64,348> (K1, stage-1 FIR decimator)", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                         "traffic": (NCU_TRAFFIC_BYTES_PER_SAMPLE_K1 * C * args.chunk * args.steps / max(k1_cnt, 1)) if (C == 4096 and args.chunk == 65536) else None,
                         "traffic_source": "ncu --set full capture of this workload, profiles/r2_k1_ncu_full_raw.csv (bytes per launch)",
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": k1_bytes, "avg_launch_ms": k1_avg_ms, "launches_timed": k1_cnt,
                         "k1_share_of_step": (k1_ms / leg["ms"]) if leg["ms"] else None, "rest_of_step_ms": (leg["rest_ms"] / leg["rest_cnt"]) if leg["rest_cnt"] else None,
                         "pipeline_gaps": leg["gaps"],
                         "step_level": {"algorithmic_bytes_per_sample": ALGO_BYTES_PER_SAMPLE_STEP, "achieved": step_gbs, "frac": step_gbs / peak,
                                        "note": "whole step (all kernels, drains and gathers of the timed region) against the same HBM peak, SURVEY 8(d)"}},
            "e2e": e2e, "gpu_launches": int(leg["launches"]), "clocks": leg["clocks"],
            "per_rank": {"ms": leg["per_rank_ms"], "host_issue_ms_per_step": leg["per_rank_issue_ms"], "host_drain_ms_per_step": leg["per_rank_drain_ms"],
                         "spread": (max(leg["per_rank_ms"]) - min(leg["per_rank_ms"])) / max(leg["per_rank_ms"]), **leg["per_rank_diag"]},
            "host_issue_ms_per_step": leg["per_rank_issue_ms"][0], "final_collect_ms": leg["final_ms"],
            "results": {"channels_gathered": args.channels, "gathers_in_timed_region": leg["gathers"], "transport": "hbd_gather_results (NCCL send/recv to rank 0)" if world > 1 else "hbd_gather_results (one rank)",
                        "chars": totals["chars"], "sentences": totals["sentences"], "sentences_min": totals["sentences_min"], "records": totals["records"],
                        "result_hash": result_hash},
            "parity": parity, "strong": strong, "wideband": wideband}

    if world == 1 and not args.no_cpu_baseline:
        from oracle import pyoracle as po
        kind = "ref" if po.available("ref") else "orc"
        try:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))
        except Exception:
            pass
        ncores = os.cpu_count() or 1
        L = synth.ring_length(FS, BAUD)
        cfg = po.make_config(baud=BAUD, dec_factor=FACTOR, record=False)
        iq = np.stack([synth.ring_iq_numpy(c, FS, BAUD, snr_db=SNR_DB) for c in range(ncores)])
        secs1, _ = po.bench(kind, cfg, iq, ncores, FS, chunk=args.chunk, reps=1)
        reps = max(1, int(args.cpu_seconds / max(secs1, 1e-3)))
        secs, chars = po.bench(kind, cfg, iq, ncores, FS, chunk=args.chunk, reps=reps)
        line["cpu_baseline"] = {"value": ncores * float(L) * reps / secs / 1e6, "unit": "MSamples/s", "cores": ncores,
                                "kind": "reference" if kind == "ref" else "port",
                                "sample": "%d threads x %d ring passes of %d samples (one reference Decoder per thread), %.1f s" % (ncores, reps, L, secs)}
    print(json.dumps(line))
    D.close()
    if parity and parity["mismatches"]:
        print("PARITY FAILURE: %d channel(s) differ from the reference Decoder" % parity["mismatches"], file=sys.stderr)
        sys.exit(3)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
