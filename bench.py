#!/usr/bin/env python
"""bench.py -- FLAC encode/decode throughput of the hot path on B200; prints one JSON result line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--streams S] [--samples L]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): float32 detector timestreams (1000, 1M) quantised with
quanta = 1e-4, full encode + decode.  One "step" = one encode pass + one decode pass over the batch
(per GPU; `--gpus N` is weak scaling: every rank owns its own (1000, 1M) shard and the only collective
is the all-gather of per-rank byte counts).

value   = raw sample bytes that went through the codec per second, 2 * raw_bytes / (t_enc + t_dec),
          whole job (all ranks), device-resident in/out, CUDA-event timed, max over ranks.
e2e     = the same metric through the public Python API (FlacArray.from_array / to_array) with
          pinned HOST buffers: H2D of the input and D2H of every result inside the timed region.
roofline= the slower of the two kernel groups: the encoder sequence (k_enc_analyze, k_enc_design, k_encode,
          k_enc_scan, k_enc_compact -- one "launch" = the sequence of one encode call) or k_dec_tile;
          algorithmic bytes (raw + compressed) per launch / CUDA-event duration (events recorded by the
          library on the launching stream around exactly those kernels).
cpu_baseline = the CPU oracle port (restatement of the reference's OpenMP-over-streams loops) timed on
          this box's host cores on a bounded sample of the same workload.
`--impl reference` times that CPU implementation as the whole job (rank 0 only).
`--dump-outputs DIR` writes what the last timed step returned on rank 0 (see dump_outputs) as DIR/<name>.npy, so
          that two builds can be compared output for output: the inputs are seeded and identical from run to run.

The benchmark writes nothing into the source tree (it may be read-only): no bytecode caches, and outputs only where
--dump-outputs points.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 123456789  # reference demo.py:12
QUANTA = 1e-4
METRIC = "encode+decode GB/s of raw samples (float32 TOD, quanta 1e-4, level 5)"


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/r02_traffic.json)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))[kernel]
        return int(t["dram_bytes_read"]) + int(t["dram_bytes_write"])
    except Exception:
        return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------
# synthetic detector timestreams: the reference's demo model (demo.py:70-97)
# ---------------------------------------------------------------------------------------------------
def make_tod_numpy(n_stream, n_samp, seed):
    rng = np.random.default_rng(seed)
    dc = 5.0 * (rng.random((n_stream, 1)) - 0.5)
    t = np.arange(n_samp)
    minf = 5 / n_samp
    wave = 2.0 * np.sin(2 * np.pi * 3 * minf * t) + 6.0 * np.sin(2 * np.pi * minf * t)
    scale = rng.random((n_stream, 1))
    out = np.empty((n_stream, n_samp), np.float32)
    for i in range(n_stream):
        out[i] = dc[i] + scale[i] * wave + rng.normal(0.0, 1.0, n_samp)
    return out


def make_tod_torch(n_stream, n_samp, seed, device):
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    dc = 5.0 * (torch.rand((n_stream, 1), generator=g, device=device) - 0.5)
    scale = torch.rand((n_stream, 1), generator=g, device=device)
    t = torch.arange(n_samp, device=device, dtype=torch.float64)
    minf = 5.0 / n_samp
    wave = (2.0 * torch.sin(2 * np.pi * 3 * minf * t) + 6.0 * torch.sin(2 * np.pi * minf * t)).to(torch.float32)
    out = torch.empty((n_stream, n_samp), dtype=torch.float32, device=device)
    chunk = max(1, (1 << 28) // n_samp)
    for i in range(0, n_stream, chunk):
        j = min(n_stream, i + chunk)
        out[i:j] = torch.randn((j - i, n_samp), generator=g, device=device)
        out[i:j] += dc[i:j] + scale[i:j] * wave
    return out


# ---------------------------------------------------------------------------------------------------
# --dump-outputs: what a caller of the timed path receives, as float32 / float64 .npy files
# ---------------------------------------------------------------------------------------------------
DUMP_ROWS = 4                 # streams whose decoded samples and compressed bytes are written
DUMP_ELEMS = 1 << 22          # cap per sampled array (16 MB as float32)
DUMP_STREAMS = 1 << 20        # cap on the per-stream arrays (24 MB for all four)


def dump_outputs(out_dir, comp, starts, nbytes, off, gain, decoded, n_stream, n_samp):
    """Write the last timed step's results: encode_device's (compressed bytes, stream starts, stream byte counts,
    offsets, gains) and decode_device's float32 samples.  Large outputs are sampled with a fixed seed, so the files
    stay below 64 MB in all and are comparable between builds: the decoded samples and compressed bytes of
    DUMP_ROWS streams (each cut to DUMP_ELEMS // DUMP_ROWS values), and the per-stream arrays of at most
    DUMP_STREAMS streams.  Bytes and integer offsets are stored as float32 / float64, which hold them exactly."""
    rng = np.random.default_rng(SEED)
    rows = np.sort(rng.choice(n_stream, min(n_stream, DUMP_ROWS), replace=False))
    per_row = DUMP_ELEMS // len(rows)
    streams = np.arange(n_stream) if n_stream <= DUMP_STREAMS else np.sort(rng.choice(n_stream, DUMP_STREAMS, replace=False))
    h_starts = starts.reshape(-1).cpu().numpy()
    h_nbytes = nbytes.reshape(-1).cpu().numpy()
    dec = decoded.reshape(n_stream, n_samp)
    pieces = [comp[int(h_starts[r]):int(h_starts[r]) + min(int(h_nbytes[r]), per_row)] for r in rows]
    arrays = {
        "decoded": dec[rows.tolist(), :min(n_samp, per_row)].cpu().numpy().astype(np.float32),
        "compressed": np.concatenate([p.cpu().numpy() for p in pieces]).astype(np.float32),
        "stream_starts": h_starts[streams].astype(np.float64),
        "stream_nbytes": h_nbytes[streams].astype(np.float64),
        "stream_offsets": off.reshape(-1).cpu().numpy()[streams].astype(np.float32),
        "stream_gains": gain.reshape(-1).cpu().numpy()[streams].astype(np.float32),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line).

    Uses NVML in-process (nvidia_ml_py) from a thread: a query costs microseconds.  (The first version
    spawned `nvidia-smi -lms 50`; with one poller per rank the driver-side cost of those queries showed up
    as tens of milliseconds of launch/sync latency in multi-GPU runs.)  Falls back to nvidia-smi.
    """
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []          # (t, sm_mhz, sm_max_mhz, set(reasons))
        self.gpu_index = gpu_index
        self.proc = None
        self.thread = None
        self.stop_flag = False
        self.t_mark = 0.0
        self.nvml = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            # torch's device index follows CUDA_VISIBLE_DEVICES; map through the UUID-free common case
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu_index
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu_index])
                except Exception:
                    idx = self.gpu_index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        R = {
            "hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8)),
            "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown",
                                           getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
            "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown",
                                           getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)),
            "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)),
        }
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        try:
            mx = float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM))
        except Exception:
            mx = 0.0
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                mask = int(get_reasons(self.handle))
                self.rows.append((time.perf_counter(), sm, mx, {k for k, b in R.items() if mask & b}))
            except Exception:
                pass
            time.sleep(0.005)

    def _read_smi(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 9:
                continue
            try:
                sm, mx = float(f[1]), float(f[2])
            except ValueError:
                continue
            rs = {name for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9])
                  if v.lower().startswith("active")}
            self.rows.append((time.perf_counter(), sm, mx, rs))

    def mark(self):
        """Only samples that arrive after this call are reported (start of the timed region)."""
        self.t_mark = time.perf_counter()

    def stop(self):
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)
        rows = [r for r in self.rows if r[0] >= self.t_mark]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(r[1] for r in rows)
        reasons = set()
        for r in rows:
            reasons |= r[3]
        busy = sm[len(sm) // 2:]  # upper half ~ samples under load
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(r[2] for r in rows)), "reasons": sorted(reasons),
                "samples": len(rows), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ---------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port (kind "port"), OpenMP over streams like compress.c:315-392
# ---------------------------------------------------------------------------------------------------
# The only numbers that come from the real libFLAC-backed reference: single-thread GB/s of raw float32 from the
# frozen notebook cells (docs/docs/cookbook.ipynb:104-136; hardware not stated), BASELINE.md section 1.
PUBLISHED_LIBFLAC = {"encode_gbs_per_thread": 0.154, "decode_gbs_per_thread": 0.895,
                     "source": "docs/docs/cookbook.ipynb:104-136 (400 MB float32, quanta 1e-7, level 5, 1 thread, CPU unspecified)"}


def honest_reference_columns(enc_gbs, dec_gbs, cores):
    """What the CPU column would read with libFLAC instead of the (slower) oracle port: per-thread figures of this run,
    the published libFLAC per-thread figures, and their perfect-scaling extrapolation to this box's cores."""
    pe, pd = PUBLISHED_LIBFLAC["encode_gbs_per_thread"], PUBLISHED_LIBFLAC["decode_gbs_per_thread"]
    est = 2.0 / (1.0 / (pe * cores) + 1.0 / (pd * cores))
    return {"per_thread_gbs": {"encode": enc_gbs / cores, "decode": dec_gbs / cores},
            "published_libflac": PUBLISHED_LIBFLAC,
            "est_libflac_same_cores": {"value": est, "unit": "GB/s", "cores": cores,
                                       "how": "published per-thread encode/decode figures x cores (perfect scaling assumed), "
                                              "combined like the metric: 2 / (1/enc + 1/dec)"}}


def cpu_pipeline(sample, threads, level=5):
    """float32 [n, L] -> seconds of (quantise, encode, decode, restore) with the reference's structure:
    converters single-threaded (utils.c has no OpenMP), encode/decode OpenMP over streams."""
    from oracle import oracle as O

    os.environ["OMP_NUM_THREADS"] = str(threads)
    try:   # the runtime may already be initialised (torchrun exports OMP_NUM_THREADS=1)
        O.lib().omp_set_num_threads(int(threads))
    except Exception:
        pass
    q = np.full(sample.shape[0], QUANTA, np.float32)
    t0 = time.perf_counter()
    ints, off, gain = O.float_to_int(sample, q)
    t1 = time.perf_counter()
    comp, starts, nbytes = O.encode(ints, level, use_threads=True)
    t2 = time.perf_counter()
    back = O.decode(comp, starts, nbytes, sample.shape[1], use_threads=True)
    t3 = time.perf_counter()
    rest = O.int_to_float(back, off, gain)
    t4 = time.perf_counter()
    assert np.array_equal(back, ints) and rest.shape == sample.shape
    return {"t_enc": t2 - t0, "t_dec": t4 - t2, "quant": t1 - t0, "encode": t2 - t1, "decode": t3 - t2,
            "restore": t4 - t3, "ratio": comp.size / sample.nbytes}


def run_reference(args):
    """--impl reference: the CPU implementation of the path on this box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O

    O.build()
    cores = os.cpu_count() or 1
    n_samp = args.samples
    per_step = max(cores, min(args.streams, 2 * cores, 128))   # bounded sample of the (streams, samples) workload
    sample = make_tod_numpy(per_step, n_samp, SEED)
    raw = sample.nbytes
    for _ in range(args.warmup):
        cpu_pipeline(sample[: max(1, min(per_step, cores))], cores)
    t_enc = t_dec = 0.0
    ratio = 0.0
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        r = cpu_pipeline(sample, cores)
        t_enc += r["t_enc"]; t_dec += r["t_dec"]; ratio = r["ratio"]
    wall = time.perf_counter() - t_wall0
    value = 2.0 * raw * args.steps / (t_enc + t_dec) / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32 (float32 in/out, double intermediates)", "data": "synthetic",
        "config": {"workload": f"float32 TOD ({args.streams}, {n_samp}) quanta=1e-4 level 5, encode+decode",
                   "sample_streams": per_step},
        "encode_gbs": raw * args.steps / t_enc / 1e9, "decode_gbs": raw * args.steps / t_dec / 1e9, "ratio": ratio,
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": cores, "kind": "port",
                         "sample": f"{per_step} of {args.streams} streams x {n_samp} float32 samples per step; "
                                   "oracle/flac_oracle.c (libFLAC absent here), OpenMP over streams, converters 1 thread"},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    line["cpu_baseline"].update(honest_reference_columns(line["encode_gbs"], line["decode_gbs"], cores))
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: flacarray_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as ge

    ge.build()
    import flacarray_b200 as fa
    from flacarray_b200 import _lib
    from flacarray_b200 import libflacarray as lf
    from flacarray_b200.mpi import TorchComm, global_bytes

    n_stream, n_samp = args.streams, args.samples
    data = make_tod_torch(n_stream, n_samp, SEED + rank, dev)
    raw = data.numel() * 4
    quanta = torch.full((n_stream,), QUANTA, dtype=torch.float32, device=dev)
    ctx = _lib.context(dev)
    comm = TorchComm() if world > 1 else None
    flat = data.reshape(-1)

    def step_device():
        comp, starts, nbytes, off, gain = lf.encode_device(flat, n_stream, n_samp, 5, quanta)
        local_nbytes = int(comp.numel())
        if comm is not None:  # the only collective on the path: byte counts -> global offsets (mpi.py:177-187)
            global_bytes(local_nbytes, starts, comm)
        mx = int(nbytes.max().item())
        out = lf.decode_device(comp, starts, nbytes, n_stream, n_samp, -1, -1, False, mx, 4096, off, gain)
        return comp, out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity guard on the exact bench input (cheap subset through the oracle) ----
    comp, out = step_device()
    ratio = comp.numel() / raw
    if rank == 0:
        from oracle import oracle as O

        sub = data[:2].cpu().numpy()
        oi, oo, og = O.float_to_int(sub, np.full(2, QUANTA, np.float32))
        want = O.int_to_float(oi, oo, og)
        got = out.reshape(n_stream, n_samp)[:2].cpu().numpy()
        if not np.array_equal(got, want):
            raise SystemExit("bench parity guard failed: GPU round trip differs from the oracle")
    del comp, out

    # ---- device-resident timed region (separate encode / decode timings inside one loop) ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.5)
    # warm-up with the same object lifetimes as the timed loop (the previous step's results are still alive
    # while the next step allocates), so that the caching allocator has reached its steady state
    comp = out = None
    for _ in range(args.warmup):
        comp, out = step_device()
    del comp, out
    ctx.profile(True)
    launches0 = ctx.launches()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    barrier()
    sampler.mark()
    t_wall0 = time.perf_counter()
    dbg = os.environ.get("FAB_BENCH_DEBUG") == "1"
    for k in range(args.steps):
        ev[k][0].record()
        th0 = time.perf_counter()
        comp, starts, nbytes, off, gain = lf.encode_device(flat, n_stream, n_samp, 5, quanta)
        th1 = time.perf_counter()
        if comm is not None:
            global_bytes(int(comp.numel()), starts, comm)
        if dbg:
            print(f"[rank {rank}] step {k}: encode_device {1e3 * (th1 - th0):.2f} ms, global_bytes "
                  f"{1e3 * (time.perf_counter() - th1):.2f} ms", file=sys.stderr, flush=True)
        ev[k][1].record()
        mx = int(nbytes.max().item())
        out = lf.decode_device(comp, starts, nbytes, n_stream, n_samp, -1, -1, False, mx, 4096, off, gain)
        ev[k][2].record()
    barrier()
    wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    launches = ctx.launches() - launches0
    if dbg:
        print(f"[rank {rank}] events: " + ", ".join(f"enc {e[0].elapsed_time(e[1]):.1f} dec {e[1].elapsed_time(e[2]):.1f}" for e in ev)
              + f" | wall {1e3 * wall:.1f} ms", file=sys.stderr, flush=True)
    t_enc = sum(e[0].elapsed_time(e[1]) for e in ev) / 1e3
    t_dec = sum(e[1].elapsed_time(e[2]) for e in ev) / 1e3
    enc_ms, enc_n = ctx.profile_ms(0)
    dec_ms, dec_n = ctx.profile_ms(1)
    ctx.profile(False)
    comp_bytes = int(comp.numel())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, comp, starts, nbytes, off, gain, out, n_stream, n_samp)
    del comp, out

    tt = torch.tensor([t_enc, t_dec, wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_enc_m, t_dec_m, wall_m = [float(x) for x in tt.cpu()]
    value = 2.0 * raw * world * args.steps / (t_enc_m + t_dec_m) / 1e9

    # ---- extra legs on one GPU: the other compression levels, and streams WITHOUT this library's frame-size table ----
    extras = {}
    if world == 1:
        ns_x = min(n_stream, 250)
        sub = data[:ns_x].reshape(-1)
        qx = quanta[:ns_x]
        lv = {}
        for level in (0, 2, 5, 8):
            best = 1e30
            for rep in range(3):
                a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
                a.record()
                c_, s_, nb_, off_, gain_ = lf.encode_device(sub, ns_x, n_samp, level, qx)
                b.record(); torch.cuda.synchronize()
                if rep:
                    best = min(best, a.elapsed_time(b))
            lv[str(level)] = {"encode_gbs": ns_x * n_samp * 4 / best / 1e6, "ratio": c_.numel() / (ns_x * n_samp * 4)}
            if level == 5:
                keep5 = (c_, s_, nb_, off_, gain_)
            del c_
        extras["levels"] = {"streams": ns_x, "by_level": lv}
        # foreign streams: the same level-5 bytes with the APPLICATION block (frame-size table "faB2") cut out, which is what
        # libFLAC would have written: fLaC + STREAMINFO (now the last metadata block) + frames.  The decoder then finds
        # the frames with its sync scan (k_dec_sync: FF F8 + header checks + CRC-8, decompress.c:274-299's job).
        c5, s5, nb5, off5, gain5 = keep5
        hs, hn = s5.cpu().numpy().reshape(-1), nb5.cpu().numpy().reshape(-1)
        nf = -(-n_samp // 4096)
        cut = 4 + 8 + 3 * nf                     # block header + "faB2" + frame count + 3 bytes per frame
        fstarts = np.zeros(ns_x, np.int64); fn = hn - cut
        fstarts[1:] = np.cumsum(fn)[:-1]
        fcomp = torch.empty(int(fn.sum()), dtype=torch.uint8, device=dev)
        for i in range(ns_x):
            a0, o0 = int(hs[i]), int(fstarts[i])
            fcomp[o0:o0 + 42] = c5[a0:a0 + 42]
            fcomp[o0 + 4] |= 0x80            # STREAMINFO is the last metadata block now
            fcomp[o0 + 42:o0 + int(fn[i])] = c5[a0 + 42 + cut:a0 + int(hn[i])]
        fs_t = torch.from_numpy(fstarts).to(dev); fn_t = torch.from_numpy(fn).to(dev)
        mxf, mx5 = int(fn.max()), int(hn.max())
        res = {}
        for name, (cc, ss, nn, mm) in {"table": (c5, s5, nb5, mx5), "foreign": (fcomp, fs_t, fn_t, mxf)}.items():
            best = 1e30
            for rep in range(3):
                a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
                a.record()
                o_ = lf.decode_device(cc, ss, nn, ns_x, n_samp, -1, -1, False, mm, 4096, off5, gain5)
                b.record(); torch.cuda.synchronize()
                if rep:
                    best = min(best, a.elapsed_time(b))
            res[name] = (best, o_)
        if not torch.equal(res["table"][1], res["foreign"][1]):
            raise SystemExit("bench: decode of the table-less streams differs from the table-indexed decode")
        extras["decode_foreign_gbs"] = ns_x * n_samp * 4 / res["foreign"][0] / 1e6
        extras["decode_table_gbs_same_sample"] = ns_x * n_samp * 4 / res["table"][0] / 1e6
        del res, fcomp, keep5, c5

    # ---- e2e: public API with pinned host buffers, H2D + D2H inside the timed region ----
    # pinned host memory per rank ~ 2.6 x the e2e array (input, compressed bytes, decoded output; the previous step's results
    # are released before the next step so the pinned pool recycles them).  The array keeps its full size at every rank
    # count as long as all ranks together stay below half of the host's available memory.
    avail = 0
    try:
        with open("/proc/meminfo") as f:
            for ln in f:
                if ln.startswith("MemAvailable:"):
                    avail = int(ln.split()[1]) * 1024
    except OSError:
        pass
    per_stream = 2.6 * n_samp * 4
    fit = int(0.5 * avail / world / per_stream) if avail else args.e2e_streams
    e2e_streams = max(16, min(n_stream, args.e2e_streams, fit))
    host = torch.empty((e2e_streams, n_samp), dtype=torch.float32, pin_memory=True)
    host.copy_(data[:e2e_streams])
    torch.cuda.synchronize()
    host_np = host.numpy()
    e2e_raw = host_np.nbytes
    # warm-up (the pinned host pool and the device pools reach their steady state)
    far = back = None
    for _ in range(3):
        del far, back
        far = fa.FlacArray.from_array(host_np, quanta=QUANTA)
        back = far.to_array()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    h2d = d2h = 0
    for _ in range(e2e_steps):
        del far, back
        far = fa.FlacArray.from_array(host_np, quanta=QUANTA)
        back = far.to_array()
        h2d += e2e_raw + far.nbytes
        d2h += far.nbytes + back.nbytes
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    te = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = 2.0 * e2e_raw * world * e2e_steps / float(te.item()) / 1e9
    # ---- the copy ceiling of this box: every rank moves the same bytes per step over PCIe (pinned memory, both directions
    #      at once, nothing else running) -- what e2e would be if the kernels and the host-side staging were free
    far_nbytes = int(far.nbytes)
    del far
    dsrc = data[:e2e_streams]
    back_t = torch.from_numpy(back) if isinstance(back, np.ndarray) else back
    pinned_out = back_t if (not back_t.is_cuda and back_t.is_pinned()) else torch.empty_like(host)
    s_up, s_dn = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    frac = far_nbytes / e2e_raw
    rows_c = max(1, int(e2e_streams * frac))          # the compressed bytes, as rows of the same buffers
    def copy_step():
        with torch.cuda.stream(s_up):
            dsrc.copy_(host, non_blocking=True)
            dsrc[:rows_c].copy_(host[:rows_c], non_blocking=True)
        with torch.cuda.stream(s_dn):
            pinned_out.view(-1)[:host.numel()].view_as(host).copy_(dsrc, non_blocking=True)
            pinned_out.view(-1)[:rows_c * n_samp].view(rows_c, n_samp).copy_(dsrc[:rows_c], non_blocking=True)
    copy_step(); barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        copy_step()
    torch.cuda.synchronize()
    t_copy = time.perf_counter() - t0
    tc = torch.tensor([t_copy], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
    copy_ceiling = 2.0 * e2e_raw * world * e2e_steps / float(tc.item()) / 1e9
    del back, back_t, pinned_out

    if rank == 0:
        peak, peak_src = measured_peak()
        alg_enc = raw + comp_bytes            # SURVEY 8(d): raw in + compressed out, per launch
        alg_dec = comp_bytes + raw
        enc_gbs = alg_enc * enc_n / (enc_ms / 1e3) / 1e9 if enc_ms > 0 else None
        dec_gbs = alg_dec * dec_n / (dec_ms / 1e3) / 1e9 if dec_ms > 0 else None
        ENC = "k_minmax+k_quant_params+k_enc_analyze+k_enc_design+k_encode+k_enc_scan+k_enc_compact+k_enc_finalize"
        dominant = ENC if (enc_ms / max(enc_n, 1)) >= (dec_ms / max(dec_n, 1)) else "k_dec_tile"
        ach = enc_gbs if dominant == ENC else dec_gbs
        # CPU baseline beside it (bounded sample, all host cores)
        cores = os.cpu_count() or 1
        cpu = None
        if not args.no_cpu_baseline:
            from oracle import oracle as O

            O.build()
            ns = max(cores, min(n_stream, 2 * cores, 128))
            sample = data[:ns].cpu().numpy()
            r = cpu_pipeline(sample, cores)
            cpu = {"value": 2.0 * sample.nbytes / (r["t_enc"] + r["t_dec"]) / 1e9, "unit": "GB/s", "cores": cores,
                   "kind": "port",
                   "sample": f"{ns} of {n_stream} streams x {n_samp} float32 samples, one pass; oracle/flac_oracle.c "
                             "(libFLAC absent), OpenMP over streams, converters single-threaded like utils.c",
                   "encode_gbs": sample.nbytes / r["t_enc"] / 1e9, "decode_gbs": sample.nbytes / r["t_dec"] / 1e9,
                   "ratio": r["ratio"]}
            cpu.update(honest_reference_columns(cpu["encode_gbs"], cpu["decode_gbs"], cores))
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * (t_enc_m + t_dec_m) / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32 (float32 in/out, double intermediates)", "data": "synthetic",
            "config": {"workload": f"float32 TOD ({n_stream}, {n_samp}) per GPU, quanta=1e-4, level 5, encode+decode",
                       "l2": "inputs (4 GB) larger than L2 (126 MB); no explicit flush",
                       "parallelism": f"streams sharded over {world} GPU(s); all-gather of byte counts only"},
            "encode_gbs": raw * world * args.steps / t_enc_m / 1e9, "decode_gbs": raw * world * args.steps / t_dec_m / 1e9,
            "ratio": ratio, "wall_ms_per_step": 1e3 * wall_m / args.steps,
            "roofline": {"bound": "hbm", "kernel": dominant, "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": (ach / peak) if ach else None,
                         "traffic": ncu_traffic("encode" if dominant == ENC else "k_dec_tile")
                         if (n_stream, n_samp) == (1000, 1000000) else None,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_enc if dominant == ENC else alg_dec,
                         "ms_per_launch": (enc_ms / max(enc_n, 1)) if dominant == ENC else (dec_ms / max(dec_n, 1))},
            "roofline_encode": {"kernel": ENC, "achieved": enc_gbs, "frac": enc_gbs / peak if enc_gbs else None,
                                "ms_per_launch": enc_ms / max(enc_n, 1)},
            "roofline_decode": {"kernel": "k_dec_tile+k_dec_crc", "achieved": dec_gbs, "frac": dec_gbs / peak if dec_gbs else None,
                                "ms_per_launch": dec_ms / max(dec_n, 1)},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "GB/s", "h2d_bytes_per_step": h2d // e2e_steps,
                    "d2h_bytes_per_step": d2h // e2e_steps, "streams": e2e_streams, "steps": e2e_steps,
                    "copy_ceiling": copy_ceiling, "frac_of_copy_ceiling": e2e_value / copy_ceiling,
                    "copy_ceiling_how": "same H2D + D2H bytes per step from / to pinned memory on two streams, all ranks at once, "
                                        "no kernels, no staging"},
            "gpu_launches": launches, "clocks": clocks,
        }
        line.update(extras)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=1000)
    ap.add_argument("--samples", type=int, default=1000000)
    ap.add_argument("--e2e-streams", type=int, default=1000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (sampled, float32/float64) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
