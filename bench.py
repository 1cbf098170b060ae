#!/usr/bin/env python
"""bench.py — resampled output Msamples/s on BASELINE.json configs[1]:
4096 stereo float streams, 44.1 -> 48 kHz, 256-tap ART filters (256 phases, Blackman-Harris,
inter-phase interpolation), 1 s of audio per stream per step, on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  `value` = whole-job output Msamples/s with inputs
resident in HBM; `e2e` = the same through the host-buffer C-ABI call (pinned host
memory, H2D + D2H inside the timed region); `roofline` = the resampler kernel against the
FP32-FMA peak measured by an FFMA-only probe in the same run (plus its HBM view);
`cpu_baseline` = the unmodified reference (oracle/_ref) or the oracle port on the host cores.
Multi-GPU: streams are sharded by index, one process per GPU, no collective on the data
path; NCCL only gathers per-rank checksums after the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the tree may be read-only: leave no __pycache__ in it
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

f32 = np.float32

# ---- the workload (BASELINE.json configs[1]; SURVEY.md §8d) ---------------------------------
STREAMS_PER_GPU = 4096
CHANNELS = 2
TAPS = 256
FILTERS = 256
FLAGS = 0x1 | 0x2  # SUBSAMPLE_INTERPOLATE | BLACKMAN_HARRIS
SRC_RATE, DST_RATE = 44100, 48000
RATIO = f32(DST_RATE) / f32(SRC_RATE)
N_IN = 44100  # 1 s per stream per step
DISTINCT = 128  # distinct synthetic streams (64 multitone + 64 noise), tiled over the batch
FLOP_PER_SAMPLE = 4 * TAPS  # two T-tap dot products, 2 flop per tap (SURVEY.md §8d)
BYTES_PER_SAMPLE = 4.0 + 4.0 / float(RATIO)  # f32 out + f32 in per output sample
WORKLOAD = ("batch of 4096 stereo streams 44.1->48 kHz, 256 taps, 256 phases, Blackman-Harris + "
            "inter-phase interpolation, 1 s (44100 frames) per stream per step")


def synth_streams(n_rows, n_in, rank=0):
    from signals import multitone, noise
    base = []
    for s in range(min(DISTINCT, n_rows)):
        sid = rank * DISTINCT + s
        base.append(multitone(n_in, CHANNELS, float(SRC_RATE), stream=sid, amp=0.5) if s % 2 == 0
                    else noise(n_in, CHANNELS, stream=sid, amp=0.5))
    base = np.stack(base)
    reps = (n_rows + base.shape[0] - 1) // base.shape[0]
    return np.tile(base, (reps, 1))[:n_rows]


class ClockSampler:
    """SM clock, power and throttle reasons of one GPU, sampled every ~20 ms by NVML in a thread
    (nvidia-smi -lms as a fallback) while the warm-up and timed steps run."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.stop_flag, self.t, self.marks = gpu_index, [], False, None, []

    def _nvml_loop(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((time.perf_counter(), float(sm), float(mx), pw, int(rs)))
            except Exception:
                pass
            time.sleep(0.02)

    def _smi_loop(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}",
                                 "--format=csv,noheader,nounits", "-lms", "100"],
                                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        bits = [0x8, 0x40, 0x20, 0x4]
        for line in proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 7:
                try:
                    rs = sum(b for b, v in zip(bits, parts[3:7]) if v.lower().startswith("active"))
                    self.rows.append((time.perf_counter(), float(parts[0]), float(parts[1]), float(parts[2]), rs))
                except ValueError:
                    pass
            if self.stop_flag:
                break
        proc.terminate()

    def start(self):
        try:
            import pynvml  # noqa: F401
            target = self._nvml_loop
        except Exception:
            target = self._smi_loop
        self.t = threading.Thread(target=target, daemon=True)
        self.t.start()

    def mark(self):
        self.marks.append(time.perf_counter())

    def stop(self):
        self.stop_flag = True
        if self.t:
            self.t.join(timeout=2)
        rows = self.rows
        timed = [r for r in rows if len(self.marks) >= 2 and self.marks[0] <= r[0] <= self.marks[1]]
        use = timed if len(timed) >= 3 else rows  # short timed regions: fall back to warm-up + timed samples
        if not use:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        pmax = max(r[3] for r in use)
        loaded = [r for r in use if r[3] >= 0.5 * pmax] or use
        reasons = set()
        for r in use:
            for bit, name in self.REASONS.items():
                if r[4] & bit:
                    reasons.add(name)
        out = {"sm_mhz": float(np.median([r[1] for r in loaded])), "sm_max_mhz": max(r[2] for r in use),
               "power_w_max": pmax, "samples": len(use), "samples_in_timed_region": len(timed),
               "window": "timed region" if use is timed else "warm-up + timed region", "reasons": sorted(reasons)}
        if len(self.marks) >= 4:  # the second timed loop (per-launch kernel events: the roofline's numerator)
            second = [r for r in rows if self.marks[2] <= r[0] <= self.marks[3]]
            if second:
                out["roofline_loop"] = {"sm_mhz": float(np.median([r[1] for r in second])),
                                        "sm_mhz_min": min(r[1] for r in second),
                                        "power_w_max": max(r[3] for r in second), "samples": len(second)}
        return out


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference_arm(n_streams, n_in, threads, reps=1):
    """Times the reference's own CPU implementation (oracle/_ref when the reference was compiled,
    else the oracle port) on `n_streams` streams of the workload.  Returns dict."""
    from oracle_lib import Oracle, Reference, have_reference
    if have_reference():
        be, kind = Reference(), "reference"
    else:
        be, kind = Oracle(), "port"
    x = synth_streams(n_streams, n_in)
    cap = int(n_in * float(RATIO)) + 64
    best, gen = None, 0
    for _ in range(reps):
        secs, gen, _ = be.bench_resample(threads, CHANNELS, TAPS, FILTERS, 1.0, FLAGS, TAPS / 2.0, x, cap, RATIO)
        best = secs if best is None else min(best, secs)
    msps = gen * CHANNELS / best / 1e6
    return {"value": msps, "unit": "Msamples/s", "cores": threads, "kind": kind, "seconds": best,
            "sample": f"{n_streams} streams x {n_in} frames of the workload ({gen * CHANNELS} output samples), "
                      f"{threads} host threads, processing time only"}


def run_reference(args, out):
    """--impl reference: the reference's CPU path on the host cores, same config/metric."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = host_threads()
    n_streams = max(threads * 16, 16)
    n_in = N_IN
    for _ in range(args.warmup):
        cpu_reference_arm(max(threads, 2), n_in // 8, threads)
    t0 = time.time()
    vals = [cpu_reference_arm(n_streams, n_in, threads) for _ in range(args.steps)]
    wall = time.time() - t0
    secs = [v["seconds"] for v in vals]
    msps = float(np.mean([v["value"] for v in vals]))
    line = {
        "impl": "reference", "metric": "resampled output Msamples/s (4096 stereo streams, 256 taps)",
        "value": msps, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * float(np.mean(secs)), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "step": vals[0]["sample"], "l2": "n/a (CPU)"},
        "cpu_baseline": {"value": msps, "unit": "Msamples/s", "cores": threads, "kind": vals[0]["kind"],
                         "sample": vals[0]["sample"]},
        "e2e": {"value": msps, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
    }
    print(json.dumps(line), file=out, flush=True)
    return 0


def protect_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries (NCCL prints its version there) write
    to fd 1 directly, so fd 1 is pointed at stderr and the JSON line goes to a private copy of stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


_ALL_CPUS = None  # the affinity mask before bind_to_gpu_cpus (the CPU baseline leg gets all cores back)


def bind_to_gpu_cpus(gpu):
    """Pin this process to the CPUs NVML reports as local to its GPU, so that the pinned host buffers of the
    end-to-end path are allocated (first touch) on the GPU's NUMA node.  Returns a note for the JSON line."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(gpu)
        global _ALL_CPUS
        _ALL_CPUS = os.sched_getaffinity(0)
        before = len(_ALL_CPUS)
        nv.nvmlDeviceSetCpuAffinity(h)
        after = len(os.sched_getaffinity(0))
        return f"nvmlDeviceSetCpuAffinity: {before} -> {after} CPUs"
    except Exception as exc:  # no NVML, no permission: run unpinned
        return f"unpinned ({type(exc).__name__})"


class Ranks:
    """Barrier / max-over-ranks / gather for one process per GPU.  N > 1 goes through the library's own C entry
    points (espb_dist_*: ncclCommInitRank + ncclAllGather over NVLink) — no torch in this file."""

    def __init__(self, espb, rank, world):
        self.espb, self.rank, self.world = espb, rank, world
        self.nccl = espb.NcclGather(rank, world) if world > 1 else None

    def barrier(self):
        L = self.espb.lib()
        self.espb.capi._check(L.espb_device_sync(), "sync")
        if self.nccl:
            self.nccl.barrier()
            self.espb.capi._check(L.espb_device_sync(), "sync")

    def max(self, v):
        return max(self.all_floats(v))

    def all_floats(self, v):
        """The value of every rank, in rank order (gathered as bit patterns by ncclAllGather)."""
        import struct
        bits = struct.unpack("<Q", struct.pack("<d", float(v)))[0]
        return [struct.unpack("<d", struct.pack("<Q", g[0]))[0] for g in self.gather([bits])]

    def gather(self, words):
        return self.nccl.allgather(words) if self.nccl else [[int(w) for w in words]]

    def close(self):
        if self.nccl:
            self.nccl.close()


def timed_steps(espb, ranks, stream, step, steps, warmup):
    """W warm-up steps, then K steps between CUDA events on `stream`, bracketed by barrier + device sync on both
    sides; returns (ms per step, max over ranks)."""
    L = espb.lib()
    dbg = os.environ.get("ESPB_BENCH_DEBUG")
    for _ in range(warmup):
        step()
    ranks.barrier()
    ev0, ev1 = L.espb_event_create(), L.espb_event_create()
    L.espb_event_record(ev0, stream)
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        if dbg:
            print(f"[bench] step enqueued in {(time.perf_counter() - t0) * 1e3:.2f} ms", file=sys.stderr)
    L.espb_event_record(ev1, stream)
    ms = espb.capi.C.c_float(0)
    espb.capi._check(L.espb_event_elapsed_ms(ev0, ev1, espb.capi.C.byref(ms)), "elapsed")
    ranks.barrier()
    L.espb_event_destroy(ev0)
    L.espb_event_destroy(ev1)
    per_rank = [t / steps for t in ranks.all_floats(float(ms.value))]
    timed_steps.per_rank = per_rank
    return max(per_rank)


def timed_wall(ranks, step, steps, warmup):
    """End-to-end legs: synchronous host-buffer calls, wall clock between barriers, max over ranks."""
    for _ in range(warmup):
        step()
    ranks.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    ranks.barrier()
    return ranks.max((time.perf_counter() - t0) / steps)


def pcm_rows(n_rows, n_samples, bits, distinct, seed, first_row=0):
    """Packed little-endian PCM rows: Gaussian noise at -12 dBFS, `distinct` different rows tiled by GLOBAL row index
    (so a sharded batch holds the same streams whatever the number of ranks)."""
    nb = (bits + 7) // 8
    rng = np.random.default_rng(seed)
    base = (rng.normal(0, 0.25, size=(distinct, n_samples)).clip(-1, 0.9999) * (2 ** (8 * nb - 1))).astype(np.int64)
    raw = np.zeros((distinct, n_samples * nb), np.uint8)
    for b in range(nb):
        raw[:, b::nb] = (base >> (8 * b)) & 0xFF
    idx = (np.arange(n_rows) + first_row) % distinct
    return raw[idx]


def link_fraction(h2d_bytes, d2h_bytes, e2e_seconds, link):
    """Time the host link alone needs for the step's bytes — the slowest of (H2D bytes at the H2D-only rate, D2H bytes
    at the D2H-only rate, all bytes at the duplex rate), rates from the link probe of this run with every rank copying
    at the same time — as a fraction of the measured end-to-end step time (1.0 = the step is nothing but the wire)."""
    if not link or not link.get("duplex_sum_gbs"):
        return None
    floor_s = max(h2d_bytes / (link["h2d_gbs"] * 1e9), d2h_bytes / (link["d2h_gbs"] * 1e9),
                  (h2d_bytes + d2h_bytes) / (link["duplex_sum_gbs"] * 1e9))
    return floor_s / e2e_seconds


# ---------------------------------------------------------------------------------------------------------------
# configs[2]: 16 kHz -> 48 kHz mono voice, art_biquad post-filter, 16384 streams, int16 in / int16 out (wrapper)
# ---------------------------------------------------------------------------------------------------------------
def bench_c3(espb, ranks, stream, peak_tf, link, steps, want_e2e, checks):
    L = espb.lib()
    ns, ch, sr, dr, bits, taps, filters, frames = 16384, 1, 16000, 48000, 16, 256, 256, 16000
    cap = frames * 3 + 64
    raw = pcm_rows(ns, frames * ch, bits, 64, 3, first_row=ranks.rank * ns)
    r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, bits, bits, ch, True, True, taps, filters)
    r.set_option(espb.OPT_PLAN_CACHE, 0)
    r.set_option(espb.OPT_KERNEL_TIMING, 1)
    in_row, out_row = raw.shape[1], (cap * ch * 2 + 15) & ~15
    d_in, d_out = espb.DeviceBuffer.from_numpy(raw), espb.DeviceBuffer(ns * out_row)
    res, calls = {}, [0]

    def step():  # steady-state streaming call: state carried from call to call, enqueued without synchronising
        res["r"] = r.resample_dev_async(d_in.ptr, in_row, d_out.ptr, out_row, frames, cap, 0.0, stream)
        calls[0] += 1

    ms = timed_steps(espb, ranks, stream, step, steps, 3)
    k_ms, k_n = r.kernel_time()
    gen = res["r"]["frames_generated"]
    samples_rank = gen * ch * ns
    k_ms_call = k_ms / max(calls[0], 1)
    tf = 4.0 * taps * samples_rank / (k_ms_call * 1e-3) / 1e12 if k_ms_call > 0 else 0.0
    rec = {"workload": "16 kHz -> 48 kHz mono voice, art_biquad post-filter (2 sections), 16384 streams per GPU, "
                       "int16 in / int16 out through espb_resampler_resample_async, 1 s (16000 frames) per step",
           "scaling": "weak", "value": samples_rank * ranks.world / (ms * 1e-3) / 1e6, "unit": "Msamples/s",
           "ms_per_step": ms, "ms_per_step_by_rank": timed_steps.per_rank, "frames_out": gen,
           "filter": r.policy()["filter"],
           "roofline": {"kernel": "espb_resample_kernel (time-major in, time-major out)", "bound": "fp32_fma",
                        "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf if peak_tf else None,
                        "kernel_ms": k_ms_call, "kernel_share_of_step": k_ms_call / ms if ms else None},
           "hbm_bytes_per_step_algorithmic": ns * (frames * 2 + gen * 2),
           "l2": "PCM in + out 2.1 GB per step >> L2"}
    if want_e2e:
        h_in = espb.PinnedBuffer(raw.size, np.uint8)
        h_in.array[:] = raw.reshape(-1)
        h_out = espb.PinnedBuffer(ns * out_row, np.uint8)
        rr = {}

        def e2e_step():
            rr["r"] = r.resample_host_ptr(h_in.ptr, in_row, h_out.ptr, out_row, frames, cap, 0.0)
            calls[0] += 1

        sec = timed_wall(ranks, e2e_step, max(3, min(steps, 6)), 2)
        g2 = rr["r"]["frames_generated"]
        nbytes = ns * (frames * 2 + g2 * 2)
        rec["e2e"] = {"value": g2 * ch * ns * ranks.world / sec / 1e6, "unit": "Msamples/s", "ms_per_step": sec * 1e3,
                      "h2d_bytes_per_step": ns * frames * 2, "d2h_bytes_per_step": ns * g2 * 2,
                      "api": "espb_resampler_resample_host (int16 PCM on the wire: half the bytes of the float call)",
                      "frac_of_link": link_fraction(ns * frames * 2, ns * g2 * 2, sec, link)}
        if checks is not None:  # the CPU leg re-computes one stream: same input `calls` times through the oracle
            row = ns - 1
            checks.append(("C3", dict(raw=raw[row].copy(), calls=calls[0], frames=frames, cap=cap, sr=sr, dr=dr,
                                      got=h_out.array.reshape(ns, out_row)[row, : g2 * 2].copy(), gen=g2), rec))
        h_in.free()
        h_out.free()
    rec["checksum"] = espb.checksum_u32(d_out.ptr, ns * out_row // 4, stream) & 0x7FFFFFFFFFFFFFFF
    r.free()
    d_in.free()
    d_out.free()
    return rec


# ---------------------------------------------------------------------------------------------------------------
# configs[3]: 96 kHz -> 44.1 kHz, 24-bit, 8 channels, 1024 taps, ONE long stream per GPU (pre-filter in time blocks)
# ---------------------------------------------------------------------------------------------------------------
def bench_c4(espb, ranks, stream, peak_tf, link, steps, want_e2e, checks):
    ns, ch, sr, dr, bits, taps, filters, seconds = 1, 8, 96000, 44100, 24, 1024, 256, 30
    frames = sr * seconds
    cap = int(frames * dr / sr) + 64
    raw = pcm_rows(ns, frames * ch, bits, 1, 4 + ranks.rank)
    in_row, out_row = raw.shape[1], (cap * ch * 3 + 15) & ~15
    d_in, d_out = espb.DeviceBuffer.from_numpy(raw), espb.DeviceBuffer(ns * out_row)
    r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, bits, bits, ch, True, True, taps, filters)
    r.set_option(espb.OPT_PLAN_CACHE, 0)
    first = r.resample_dev(d_in.ptr, in_row, d_out.ptr, out_row, frames, cap, 0.0, stream)  # fresh state: checked below
    head = d_out.download(np.uint8, 44100 * ch * 3)
    r.set_option(espb.OPT_KERNEL_TIMING, 1)
    res, calls = {}, [0]

    def step():
        res["r"] = r.resample_dev_async(d_in.ptr, in_row, d_out.ptr, out_row, frames, cap, 0.0, stream)
        calls[0] += 1

    ms = timed_steps(espb, ranks, stream, step, steps, 3)
    k_ms, k_n = r.kernel_time()
    gen = res["r"]["frames_generated"]
    samples_rank = gen * ch * ns
    k_ms_call = k_ms / max(calls[0], 1)
    tf = 4.0 * taps * samples_rank / (k_ms_call * 1e-3) / 1e12 if k_ms_call > 0 else 0.0
    repaired, warm = r.biquad_block_stats()
    rec = {"workload": f"96 kHz -> 44.1 kHz, 8 channels, 24-bit in / out, 1024 taps, art_biquad pre-filter, ONE stream "
                       f"per GPU, {seconds} s ({frames} frames) per step (replicas only: a stream does not shard)",
           "scaling": "replicas", "value": samples_rank * ranks.world / (ms * 1e-3) / 1e6, "unit": "Msamples/s",
           "ms_per_step": ms, "ms_per_step_by_rank": timed_steps.per_rank, "frames_out": gen,
           "filter": r.policy()["filter"], "realtime_factor": seconds / (ms * 1e-3),
           "biquad": {"mode": "time blocks of 8192 frames, hand-over verified on the device (exact by construction)",
                      "blocks_repaired": repaired, "warmup_rows": warm},
           "roofline": {"kernel": "espb_resample_fs_kernel<SV=8,B=2> (few-series form: lanes own outputs)",
                        "bound": "shared-memory wavefronts (FP32 FMA peak as the denominator)", "achieved": tf,
                        "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf if peak_tf else None,
                        "kernel_ms": k_ms_call, "kernel_share_of_step": k_ms_call / ms if ms else None},
           "l2": "PCM in 69 MB per step, but every stage streams the time-major staging rows (2 x 1.5 GB) >> L2"}
    if want_e2e:
        h_in = espb.PinnedBuffer(raw.size, np.uint8)
        h_in.array[:] = raw.reshape(-1)
        h_out = espb.PinnedBuffer(ns * out_row, np.uint8)
        rr = {}

        def e2e_step():
            rr["r"] = r.resample_host_ptr(h_in.ptr, in_row, h_out.ptr, out_row, frames, cap, 0.0)

        sec = timed_wall(ranks, e2e_step, 3, 1)
        g2 = rr["r"]["frames_generated"]
        rec["e2e"] = {"value": g2 * ch * ns * ranks.world / sec / 1e6, "unit": "Msamples/s", "ms_per_step": sec * 1e3,
                      "h2d_bytes_per_step": ns * frames * ch * 3, "d2h_bytes_per_step": ns * g2 * ch * 3,
                      "api": "espb_resampler_resample_host (24-bit PCM on the wire)",
                      "frac_of_link": link_fraction(ns * frames * ch * 3, ns * g2 * ch * 3, sec, link)}
        h_in.free()
        h_out.free()
    if checks is not None:  # first second of the first (fresh-state) call against the composed CPU pipeline
        checks.append(("C4", dict(raw=raw[0, : 96000 * ch * 3].copy(), head=head, pol=r.policy(), ch=ch, taps=taps,
                                  filters=filters), rec))
    rec["first_call_frames"] = first["frames_generated"]
    rec["checksum"] = espb.checksum_u32(d_out.ptr, ns * out_row // 4, stream) & 0x7FFFFFFFFFFFFFFF
    r.free()
    d_in.free()
    d_out.free()
    return rec


# ---------------------------------------------------------------------------------------------------------------
# configs[4]: 65536 stereo float streams 48 kHz -> 44.1 kHz, sharded by stream index over the ranks (STRONG scaling)
# ---------------------------------------------------------------------------------------------------------------
def bench_c5(espb, ranks, stream, peak_tf, link, steps, want_e2e, checks):
    L = espb.lib()
    total, ch, taps, filters, flags = 65536, 2, 256, 256, 0x1
    ratio = f32(44100) / f32(48000)
    lowpass = float(ratio * f32(0.96))
    chunk, calls_per_step = 6000, 8  # 1 s per stream per step as 8 streaming calls of 0.125 s (bounded memory)
    first, ns = espb.shard_range(total, ranks.rank, ranks.world)
    cap = int(chunk * float(ratio)) + 64
    in_row, out_row = chunk * ch, cap * ch
    from signals import multitone, noise
    base = np.stack([multitone(chunk, ch, 48000.0, stream=s, amp=0.5) if s % 2 == 0
                     else noise(chunk, ch, stream=s, amp=0.5) for s in range(DISTINCT)])
    idx = (np.arange(ns) + first) % DISTINCT  # by GLOBAL stream index: the same batch for every N
    h_in = espb.PinnedBuffer(ns * in_row, f32)
    h_in.array.reshape(ns, in_row)[:] = base[idx]
    d_in, d_out = espb.DeviceBuffer(ns * in_row * 4), espb.DeviceBuffer(ns * out_row * 4)
    espb.capi._check(L.espb_memcpy_h2d(d_in.ptr, h_in.ptr, ns * in_row * 4, stream), "h2d")
    d_out.zero(stream)
    ctx = espb.ResampleBatch(ns, ch, taps, filters, lowpass, flags)
    ctx.set_option(espb.OPT_PLAN_CACHE, 0)
    out = {}

    def step():
        ctx.reset(stream)
        ctx.advance(taps / 2.0)
        g = 0
        for _ in range(calls_per_step):
            u, gg = ctx.process_interleaved_dev(d_in.ptr, in_row, chunk, d_out.ptr, out_row, cap, ratio, stream)
            g += gg
        out["gen"], out["last"] = g, gg

    ms = timed_steps(espb, ranks, stream, step, steps, 3)
    ms_by_rank = timed_steps.per_rank
    # the kernel alone, from its own CUDA events, in a second loop (kernel timing switches the staging overlap off)
    ctx.set_option(espb.OPT_KERNEL_TIMING, 1)
    ms_serial = timed_steps(espb, ranks, stream, step, steps, 1)
    k_ms, k_n = ctx.kernel_time()
    ctx.set_option(espb.OPT_KERNEL_TIMING, 0)
    gen = out["gen"]
    samples_rank = gen * ch * ns
    k_ms_step = k_ms / (steps + 1)
    tf = 4.0 * taps * samples_rank / (k_ms_step * 1e-3) / 1e12 if k_ms_step > 0 else 0.0
    # per-stream checksums are order independent, so the sum over ranks must not depend on N
    checksum = espb.checksum_u32(d_out.ptr, ns * out_row, stream)  # wrapping 64-bit sum: adds up over shards
    g = ranks.gather([checksum, gen, first, ns])
    assert [x[2] for x in g] == [espb.shard_range(total, r, ranks.world)[0] for r in range(ranks.world)]
    assert sum(x[3] for x in g) == total
    rec = {"workload": "65536 stereo float streams 48 kHz -> 44.1 kHz, 256 taps, ART low-pass 0.96 x ratio, sharded "
                       "by stream index over the ranks; 1 s per stream per step as 8 streaming calls of 6000 frames",
           "scaling": "strong", "streams_total": total, "streams_per_rank": ns,
           "value": gen * ch * total / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms,
           "ms_per_step_by_rank": ms_by_rank, "frames_out_per_step": gen,
           "roofline": {"kernel": "espb_resample_kernel<BPP=4,STAGES=2,CHUNK_ROWS=32>", "bound": "fp32_fma",
                        "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf if peak_tf else None,
                        "kernel_ms_per_step": k_ms_step,
                        "kernel_share_of_step": k_ms_step / ms_serial if ms_serial else None,
                        "step_ms_without_overlap": ms_serial},
           "checksums": [x[0] for x in g], "checksum_of_checksums": espb.combine_checksums([x[0] for x in g]),
           "gather": "ncclAllGather of {checksum, frames, first stream, streams} per rank through espb_dist_allgather_u64"
                     if ranks.world > 1 else "single rank",
           "l2": "input + output 12 GB per step over all ranks >> L2"}
    if want_e2e:
        h_out = espb.PinnedBuffer(ns * out_row, f32)
        rr = {}

        def e2e_step():
            ctx.reset(None)
            ctx.advance(taps / 2.0)
            gsum = 0
            for _ in range(calls_per_step):
                u, gg = ctx.process_interleaved_host(h_in.ptr, in_row, chunk, h_out.ptr, out_row, cap, ratio)
                gsum += gg
            rr["gen"], rr["last"] = gsum, gg

        sec = timed_wall(ranks, e2e_step, 2, 1)
        nbytes = ns * (calls_per_step * in_row * 4 + rr["gen"] * ch * 4)
        rec["e2e"] = {"value": rr["gen"] * ch * total / sec / 1e6, "unit": "Msamples/s", "ms_per_step": sec * 1e3,
                      "h2d_bytes_per_step": ns * calls_per_step * in_row * 4, "d2h_bytes_per_step": ns * rr["gen"] * ch * 4,
                      "api": "espb_resampleProcessInterleavedHost, 8 calls per step",
                      "frac_of_link": link_fraction(ns * calls_per_step * in_row * 4, ns * rr["gen"] * ch * 4, sec, link)}
        if checks is not None:
            row = ns - 1
            checks.append(("C5", dict(x=h_in.array.reshape(ns, in_row)[row].copy(), calls=calls_per_step, cap=cap,
                                      ratio=ratio, lowpass=lowpass, flags=flags, taps=taps, filters=filters,
                                      got=h_out.array.reshape(ns, out_row)[row, : rr["last"] * ch].copy(),
                                      gen=rr["last"]), rec))
        h_out.free()
    ctx.free()
    h_in.free()
    d_in.free()
    d_out.free()
    return rec


DUMP_STREAMS = 64  # 64 streams x 95726 output samples x 4 bytes = 24.5 MB per dump


def dump_outputs(espb, path, d_out, out_row, ns, used, gen, stream):
    """What a caller of the timed path holds after its last step: the frame counts and the output of a fixed, seeded
    sample of this rank's streams, as .npy files (float32 samples, float64 counts and stream indices), so that two
    builds can be compared output for output on the same inputs."""
    L = espb.lib()
    rows = np.sort(np.random.default_rng(0).choice(ns, size=min(ns, DUMP_STREAMS), replace=False))
    y = np.empty((rows.size, gen * CHANNELS), f32)
    for k, r in enumerate(rows):
        espb.capi._check(L.espb_memcpy_d2h(y[k].ctypes.data, d_out.ptr + int(r) * out_row * 4, y[k].nbytes, stream),
                         "d2h")
    espb.capi._check(L.espb_stream_sync(stream), "sync")
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "output.npy"), y)
    np.save(os.path.join(path, "output_streams.npy"), rows.astype(np.float64))
    np.save(os.path.join(path, "frames_used_generated.npy"), np.array([used, gen], np.float64))


def run_checks(checks, mode):
    """CPU leg (rank 0, N = 1): one stream of every sub-record re-computed by the CPU restatement of the reference."""
    from oracle_lib import Oracle
    orc = Oracle()
    tol = 0.0 if mode == "exact" else 1e-6
    for name, c, rec in checks:
        if name == "C3":  # fast mode: PCM codes may differ by 1 LSB where the float result sits on a rounding edge
            w = orc.wrapper(c["frames"], c["cap"], float(c["sr"]), float(c["dr"]), 16, 16, 1)
            for _ in range(c["calls"]):
                yo, ro = w.resample(c["raw"], c["frames"], c["cap"], 0.0)
            assert ro["frames_generated"] == c["gen"], (name, ro["frames_generated"], c["gen"])
            d = np.abs(c["got"].view(np.int16).astype(np.int64) - yo.view(np.int16).astype(np.int64))
            if int(d.max()) > 1:
                raise SystemExit(f"bench.py: {name} parity check failed (max PCM code difference {int(d.max())})")
            rec["parity_vs_oracle"] = {"max_lsb": int(d.max()), "codes_differing": float((d > 0).mean()),
                                       "stream_calls_replayed": c["calls"]}
        elif name == "C4":
            from oracle_lib import Oracle as _O  # noqa: F401
            ch, taps, pol = c["ch"], c["taps"], c["pol"]
            xf = orc.quantized_to_float(c["raw"], 96000 * ch, 24, 0.0)
            if pol["filter"] == "pre":
                for k in range(ch):
                    for _ in range(2):
                        orc.biquad(pol["coeffs"], 1.0).apply_buffer(xf[k:], ch, n=96000)
            o = orc.resampler(ch, taps, c["filters"], float(pol["art_lowpass"]), pol["art_flags"])
            o.advance(taps / 2.0)
            yf, used, gen = o.process_interleaved(xf, 44200, pol["sample_ratio"])
            q, _ = orc.float_to_quantized(np.ascontiguousarray(yf), 24)
            n = (gen - 600) * ch * 3  # the one-second CPU run lacks the frames after it: compare what both know
            a = np.frombuffer(c["head"][:n].tobytes(), np.uint8).reshape(-1, 3).astype(np.int64)
            b = np.frombuffer(q[:n].tobytes(), np.uint8).reshape(-1, 3).astype(np.int64)
            va = a[:, 0] | (a[:, 1] << 8) | (a[:, 2] << 16)
            vb = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
            d = np.abs(((va ^ 0x800000) - 0x800000) - ((vb ^ 0x800000) - 0x800000))
            if int(d.max()) > 8:  # 1e-6 full scale = 8.4 codes at 24 bits
                raise SystemExit(f"bench.py: {name} parity check failed (max PCM code difference {int(d.max())})")
            rec["parity_vs_oracle"] = {"max_lsb_24bit": int(d.max()), "codes_differing": float((d > 0).mean()),
                                       "frames_compared": gen - 600}
        elif name == "C5":
            o = orc.resampler(2, c["taps"], c["filters"], c["lowpass"], c["flags"])
            o.advance(c["taps"] / 2.0)
            for _ in range(c["calls"]):
                yo, uo, go = o.process_interleaved(c["x"], c["cap"], c["ratio"])
            err = float(np.max(np.abs(c["got"].astype(np.float64) - yo[: go * 2])))
            if go != c["gen"] or err > tol:
                raise SystemExit(f"bench.py: {name} parity check failed (generated {c['gen']} vs {go}, max-abs {err})")
            rec["parity_vs_oracle"] = {"max_abs": err, "calls_replayed": c["calls"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=STREAMS_PER_GPU, help="streams per GPU (default: the metric's 4096)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3 / C4 / C5 sub-records")
    ap.add_argument("--configs", default="C5,C3,C4", help="which sub-records to run (comma-separated)")
    ap.add_argument("--mode", default="fast", choices=["fast", "exact"],
                    help="arithmetic of the dot products: fast = FFMA2 chain (the metric), exact = un-fused, bit-exact")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (a fixed sample of its streams) as DIR/*.npy")
    args = ap.parse_args()
    out = protect_stdout()
    if args.impl == "reference":
        return run_reference(args, out)
    if args.warmup < 3:
        args.warmup = 3  # timing rule: at least 3 warm-up steps

    import esp_audio_libs_b200 as espb

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if espb.device_count() <= 0:
        raise SystemExit("bench.py: no GPU and no CPU fallback (use --impl reference for the CPU arm)")
    espb.set_device(local_rank)
    info = espb.device_info()
    L = espb.lib()
    host_affinity = bind_to_gpu_cpus(local_rank)  # before the pinned buffers are allocated and touched
    ranks = Ranks(espb, rank, world)  # N > 1: ncclCommInitRank through the library's C entry points

    ns = args.streams
    cap = int(N_IN * float(RATIO)) + 64
    in_row, out_row = N_IN * CHANNELS, cap * CHANNELS

    # ---- synthetic input in pinned host memory, then resident in HBM
    x = synth_streams(ns, N_IN, rank)  # rank r owns global streams [r*ns, (r+1)*ns)
    h_in = espb.PinnedBuffer(ns * in_row, f32)
    h_in.array[:] = x.reshape(-1)
    del x
    h_out = espb.PinnedBuffer(ns * out_row, f32)
    d_in = espb.DeviceBuffer(ns * in_row * 4)
    d_out = espb.DeviceBuffer(ns * out_row * 4)
    stream = L.espb_stream_create()
    espb.capi._check(L.espb_memcpy_h2d(d_in.ptr, h_in.ptr, ns * in_row * 4, stream), "h2d")
    d_out.zero(stream)
    espb.capi._check(L.espb_stream_sync(stream), "sync")

    # ---- FP32 FMA peak of this device, measured now (roofline denominator)
    fma_tflops, fma_clock = espb.measure_fp32_fma_peak()  # best of the scalar FFMA and packed FFMA2 probes
    fma_scalar, fma_packed = espb.measure_fp32_fma_peak2()
    tile_tf = espb.measure_fp32_tile_pattern()

    ctx = espb.ResampleBatch(ns, CHANNELS, TAPS, FILTERS, 1.0, FLAGS,
                             mode=espb.MODE_EXACT if args.mode == "exact" else espb.MODE_FAST)
    ctx.set_option(espb.OPT_PLAN_CACHE, 0)  # every step re-plans: schedule, upload and expansion are timed
    st = {}

    def step():
        ctx.reset(stream)
        ctx.advance(TAPS / 2.0)  # zero delay, as resampler.cpp:94 does
        st["r"] = ctx.process_interleaved_dev(d_in.ptr, in_row, N_IN, d_out.ptr, out_row, cap, RATIO, stream)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step()
    ranks.barrier()

    ev0, ev1 = L.espb_event_create(), L.espb_event_create()
    launches0 = espb.launch_count()
    ranks.barrier()
    sampler.mark()
    L.espb_event_record(ev0, stream)
    for _ in range(args.steps):
        step()
    L.espb_event_record(ev1, stream)
    ms = espb.capi.C.c_float(0)
    espb.capi._check(L.espb_event_elapsed_ms(ev0, ev1, espb.capi.C.byref(ms)), "elapsed")
    ranks.barrier()
    sampler.mark()
    used, gen = st["r"]
    launches = espb.launch_count() - launches0
    total_ms = ranks.max(float(ms.value))  # device-timed, max over ranks (gathered by ncclAllGather)
    if args.dump_outputs and rank == 0:  # before the second loop below overwrites d_out
        dump_outputs(espb, args.dump_outputs, d_out, out_row, ns, used, gen, stream)

    # ---- second timed loop, same steps, with CUDA events around every launch of the resampler kernel (the roofline's
    # numerator).  In the loop above the kernel starts while the staging kernel is still running (programmatic
    # dependent launch), so events on the stream cannot bracket it there; with kernel timing on the library runs the
    # two back to back, and this loop also shows what the overlap is worth (`step_ms_without_overlap`).
    ctx.set_option(espb.OPT_KERNEL_TIMING, 1)
    step()
    ctx.kernel_time()  # drop the warm-up record
    ranks.barrier()
    sampler.mark()
    L.espb_event_record(ev0, stream)
    for _ in range(args.steps):
        step()
    L.espb_event_record(ev1, stream)
    espb.capi._check(L.espb_event_elapsed_ms(ev0, ev1, espb.capi.C.byref(ms)), "elapsed")
    ranks.barrier()
    sampler.mark()
    kernel_ms, kernel_launches = ctx.kernel_time()
    serial_ms_per_step = float(ms.value) / args.steps
    ctx.set_option(espb.OPT_KERNEL_TIMING, 0)
    clocks = sampler.stop() if rank == 0 else None

    samples_per_step_rank = gen * CHANNELS * ns
    samples_per_step = samples_per_step_rank * world
    ms_per_step = total_ms / args.steps
    value = samples_per_step / (ms_per_step * 1e-3) / 1e6

    # ---- correctness guard inside the bench: a sampled stream against the oracle, checksum for the gather
    checksum = espb.checksum_u32(d_out.ptr, ns * out_row, stream) & 0x7FFFFFFFFFFFFFFF
    first_stream, _ = espb.shard_range(ns * world, rank, world)
    # NCCL: the only collective, outside the timed region — per-rank checksum, frames, first stream index
    gathered = ranks.gather([checksum, gen, first_stream])
    checksums = [g[0] for g in gathered]
    assert [g[2] for g in gathered] == [espb.shard_range(ns * world, r, world)[0] for r in range(world)]

    # ---- roofline of the dominant kernel (espb_resample_kernel), from its own CUDA events
    k_ms = kernel_ms / max(kernel_launches, 1)
    flops_per_launch = FLOP_PER_SAMPLE * samples_per_step_rank * (args.steps / max(kernel_launches, 1))
    achieved_tf = flops_per_launch / (k_ms * 1e-3) / 1e12 if k_ms > 0 else 0.0
    bytes_per_launch = BYTES_PER_SAMPLE * samples_per_step_rank * (args.steps / max(kernel_launches, 1))
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peaks = json.load(fh)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None  # dram bytes per launch of the dominant kernel, from the committed ncu capture
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as fh:
                traffic = json.load(fh)
            break
        except Exception:
            pass
    roofline = {
        "kernel": "espb_resample_kernel<BPP=4,STAGES=2,CHUNK_ROWS=32,EXACT=false,TMCAP=false>", "bound": "fp32_fma", "achieved": achieved_tf,
        "peak": fma_tflops, "unit": "TFLOP/s", "frac": achieved_tf / fma_tflops if fma_tflops else None,
        "peak_source": "FMA-only probes (espb_measure_fp32_fma_peak: best of scalar FFMA and packed FFMA2) on this "
                       "GPU in this run; nominal 148 SM x 128 lanes x 2 x 1.965 GHz = 74.4",
        "peak_probe_ffma_tflops": fma_scalar, "peak_probe_ffma2_tflops": fma_packed,
        "peak_implied_sm_mhz": fma_clock,
        # the kernel's inner loop alone (register tile fed from shared memory at the kernel's occupancy; no TMA,
        # barriers or epilogue): the practical ceiling of this loop structure, for reading `frac`
        "inner_loop_probe_tflops": tile_tf,
        "frac_of_inner_loop_probe": achieved_tf / tile_tf if tile_tf else None,
        "traffic": (traffic or {}).get("dram_bytes_per_launch") if ns == STREAMS_PER_GPU else None,
        "traffic_source": (traffic or {}).get("source"),
        "algorithmic_bytes_per_launch": bytes_per_launch,
        "flop_per_sample": FLOP_PER_SAMPLE, "kernel_ms": k_ms,
        "kernel_share_of_step": k_ms * (kernel_launches / args.steps) / serial_ms_per_step,
        "measured_in": "a second timed loop of the same steps with the staging overlap off (events must bracket the "
                       "kernel alone); its step time is step_ms_without_overlap, the headline loop's is ms_per_step",
        "step_ms_without_overlap": serial_ms_per_step,
        "step_level_frac": (FLOP_PER_SAMPLE * samples_per_step_rank / (ms_per_step * 1e-3) / 1e12) / fma_tflops
        if fma_tflops else None,
        "hbm": {"achieved_gbs": bytes_per_launch / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0, "peak_gbs": hbm_peak,
                "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6.65 TB/s",
                "bytes_per_sample": BYTES_PER_SAMPLE},
    }

    # ---- the host link as plain pinned cudaMemcpyAsync sees it, every rank copying at the same time
    link = None
    if not args.no_e2e:
        ranks.barrier()
        # (1.5 GiB per direction, the size of the step's own buffers: smaller probes partly run out of the host's
        # last-level cache and overstate what a sustained stream gets)
        # every rank runs the SAME pattern at the same time: buffers are page-locked first (that takes a second and
        # differs from rank to rank), then each timed run starts on a barrier; median of 3 runs per pattern
        C = espb.capi.C
        probe = L.espb_link_probe_create(1536 << 20, 64 << 20)
        if not probe:
            raise SystemExit("bench.py: link probe allocation failed")
        rates = []
        for pattern in (0, 1, 2):
            seen = []
            for _rep in range(4):
                ranks.barrier()
                v = C.c_double(0)
                espb.capi._check(L.espb_link_probe_run(probe, pattern, C.byref(v), None), "link probe")
                seen.append(float(v.value))
            rates.append(sorted(seen[1:])[1])
        L.espb_link_probe_free(probe)
        ranks.barrier()
        link = {"h2d_gbs": rates[0], "d2h_gbs": rates[1], "duplex_each_gbs": rates[2], "duplex_sum_gbs": 2 * rates[2],
                "bytes_per_direction": 1536 << 20, "slab_bytes": 64 << 20,
                "all_ranks_duplex_sum_gbs": sum(ranks.all_floats(2 * rates[2])),
                "what": "pinned cudaMemcpyAsync, 64 MiB slabs: H2D alone, D2H alone, both at once, on this rank's GPU "
                        f"while the other {world - 1} rank(s) run the same pattern at the same time (a barrier before "
                        "each); GB/s of this rank"}

    # ---- end to end: host buffers through the public C-ABI call, H2D + D2H inside the timed region
    e2e, e2e_last = None, None
    if not args.no_e2e:
        rr = {}

        def e2e_step():
            ctx.reset(None)
            ctx.advance(TAPS / 2.0)
            rr["r"] = ctx.process_interleaved_host(h_in.ptr, in_row, N_IN, h_out.ptr, out_row, cap, RATIO)

        k = max(3, min(args.steps, 10))
        e2e_s = timed_wall(ranks, e2e_step, k, 2)  # synchronous calls: each returns after the D2H of its results
        u2, g2 = rr["r"]
        e2e_bytes = ns * in_row * 4 + ns * g2 * CHANNELS * 4
        e2e = {"value": g2 * CHANNELS * ns * world / e2e_s / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": ns * in_row * 4, "d2h_bytes_per_step": ns * g2 * CHANNELS * 4,
               "ms_per_step": e2e_s * 1e3, "steps": k,
               "api": "espb_resampleProcessInterleavedHost (pinned host buffers, 3-stream slab pipeline)",
               "link_gbs_this_rank": e2e_bytes / e2e_s / 1e9, "link_probe": link,
               "frac_of_link": link_fraction(ns * in_row * 4, ns * g2 * CHANNELS * 4, e2e_s, link)}
        e2e_last = (g2, ns - 1)  # checked against the CPU reference in the cpu_baseline leg below
    ctx.free()
    d_in.free()
    d_out.free()

    # ---- the other BASELINE configs as sub-records (their own roofline view, e2e and oracle spot-check)
    configs, checks = {}, ([] if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None)
    if not args.no_configs and ns == STREAMS_PER_GPU:
        sub_steps = max(3, min(args.steps, 5))
        for name, fn in (("C5", bench_c5), ("C3", bench_c3), ("C4", bench_c4)):
            if name in args.configs.split(","):
                configs[name] = fn(espb, ranks, stream, fma_tflops, link, sub_steps, not args.no_e2e, checks)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if _ALL_CPUS:
            os.sched_setaffinity(0, _ALL_CPUS)
        threads = host_threads()
        cb = cpu_reference_arm(threads * 8, N_IN, threads)
        one = cpu_reference_arm(2, N_IN, 1)
        cpu_baseline = {"value": cb["value"], "unit": "Msamples/s", "cores": threads, "kind": cb["kind"],
                        "sample": cb["sample"], "one_core_value": one["value"]}
        if e2e is not None:
            # the same leg doubles as the checker of what the end-to-end call brought back to the host: one stream
            # recomputed by the CPU restatement (the only other use of oracle/ in this file)
            from oracle_lib import Oracle
            g2, row = e2e_last
            o = Oracle().resampler(CHANNELS, TAPS, FILTERS, 1.0, FLAGS)
            o.advance(TAPS / 2.0)
            yo, _, go = o.process_interleaved(h_in.array[row * in_row:(row + 1) * in_row], cap, RATIO)
            got = h_out.array[row * out_row: row * out_row + g2 * CHANNELS]
            err = float(np.max(np.abs(got.astype(np.float64) - yo)))
            if go != g2 or err > (0.0 if args.mode == "exact" else 1e-6):
                raise SystemExit(f"bench.py: parity check failed (generated {g2} vs {go}, max-abs {err})")
            e2e["parity_max_abs_vs_oracle"] = err
        if checks:
            run_checks(checks, args.mode)

    if rank == 0:
        line = {
            "metric": "resampled output Msamples/s (4096 stereo streams, 256 taps)",
            "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "streams_per_gpu": ns, "channels": CHANNELS, "taps": TAPS,
                       "filters": FILTERS, "ratio": float(RATIO), "frames_in": N_IN, "frames_out": gen,
                       "mode": ("fast (tap-order FMA chain per accumulator, packed FFMA2; <=1e-6 of the reference)"
                                if args.mode == "fast" else
                                "exact (tap-order FMUL+FADD per accumulator: bit-exact with the reference)"),
                       "signals": f"{DISTINCT} distinct streams (multitone + uniform noise, A=0.5) tiled",
                       "parallelism": f"streams sharded by index over {world} GPU(s), no data-path collective",
                       "collective": ("one ncclAllGather of 3 words per rank through the library's C entry points "
                                      "(espb_dist_allgather_u64), outside the timed region" if world > 1 else "none"),
                       "l2": "inputs+outputs 3.0 GB per step >> 126 MB L2 (no flush needed)",
                       "timed_region": "per step: reset, host schedule, table upload, coefficient expansion, "
                                       "resampler kernel, history carry (plan cache off)"},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "host_affinity": host_affinity, "gpu_launches": int(launches),
            "clocks": clocks, "checksums": checksums, "checksum_of_checksums": espb.combine_checksums(checksums), "device": info["name"], "sm_count": info["sm_count"],
            "nccl_version": int(L.espb_nccl_version()), "configs": configs,
        }
        print(json.dumps(line), file=out, flush=True)
    ranks.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
