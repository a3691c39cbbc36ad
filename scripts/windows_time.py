"""Time of per-stream sample windows (FlacArray.to_windows) on the configs[1] shape.

    python scripts/windows_time.py [--streams 1000] [--samples 1000000] [--reps 21] [--out FILE]

float32 (streams, samples) detector timestreams (bench.make_tod_torch), quanta 1e-4, level 5, compressed bytes on the
device.  Cases, window starts drawn with a fixed seed:
  (a) one 10 000-sample window per stream      (+ the same windows from host-resident bytes, + the far[s, a:b] loop)
  (b) 16 windows of 1 000 samples per stream
  (c) one 100-sample window per stream
For each: median / min / max of `reps` synchronised calls after a warm-up, frames touched, and (bytes of the touched
frames + output bytes) / median time.  The full to_array() decode is timed the same way.  Every window is checked
against the full decode.  Prints one JSON object per line (and writes them to --out); the first line names the GPU and
its power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def frame_sizes(buf):
    """Frame byte sizes from the faB2 table of one stream of this library (None without one)."""
    pos = 4
    while pos + 4 <= buf.size:
        last, typ = buf[pos] >> 7, buf[pos] & 0x7F
        ln = (int(buf[pos + 1]) << 16) | (int(buf[pos + 2]) << 8) | int(buf[pos + 3])
        pos += 4
        if typ == 2 and bytes(buf[pos:pos + 4]) == b"faB2":
            cnt = int.from_bytes(bytes(buf[pos + 4:pos + 8]), "big")
            t = buf[pos + 8:pos + 8 + 3 * cnt].astype(np.int64).reshape(cnt, 3)
            return (t[:, 0] << 16) | (t[:, 1] << 8) | t[:, 2]
        pos += ln
        if last:
            break
    return None


def touched(h_comp, starts, nbytes, streams, first, last, bs=4096):
    """(frames, compressed bytes of those frames) the windows touch, each distinct frame counted once."""
    frames, fbytes = 0, 0
    sizes = {}
    seen = set()
    for s, a, b in zip(streams, first, last):
        if b <= a:
            continue
        s = int(s)
        if s not in sizes:
            sizes[s] = frame_sizes(h_comp[int(starts[s]):int(starts[s]) + int(nbytes[s])])
        for j in range(int(a) // bs, (int(b) - 1) // bs + 1):
            if (s, j) in seen:
                continue
            seen.add((s, j))
            frames += 1
            fbytes += int(sizes[s][j])
    return frames, fbytes


def timed(fn, reps, warmup=2):
    import torch

    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(min(ts)), float(max(ts))


def gpu_info():
    import torch

    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        info["nvidia_smi"] = q
    except Exception as e:  # noqa: BLE001
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1000)
    ap.add_argument("--samples", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--loop-reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=20261020)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import bench
    import flacarray_b200 as fa

    if not torch.cuda.is_available():
        raise SystemExit("windows_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    emit(dict(gpu_info(), streams=args.streams, samples=args.samples, dtype="float32", quanta=1e-4, level=5))
    ns, n = args.streams, args.samples
    x = bench.make_tod_torch(ns, n, 1, dev)
    far = fa.FlacArray.from_array(x, quanta=np.full(ns, 1e-4, np.float32), level=5)
    del x
    full = far.to_array()
    h_comp = far.compressed.cpu().numpy()
    starts = np.asarray(far.stream_starts).reshape(-1)
    nbytes = np.asarray(far.stream_nbytes).reshape(-1)
    rng = np.random.default_rng(args.seed)

    med, lo, hi = timed(lambda: far.to_array(), max(5, args.reps // 4))
    emit(dict(case="full to_array()", ms_median=med, ms_min=lo, ms_max=hi, output_bytes=ns * n * 4))

    cases = {
        "a": (np.arange(ns), 10000),
        "b": (np.repeat(np.arange(ns), 16), 1000),
        "c": (np.arange(ns), 100),
    }
    for name, (streams, length) in cases.items():
        first = rng.integers(0, n - length + 1, streams.size)
        last = first + length
        data, offs = far.to_windows(streams, first, last)
        got = data.cpu().numpy()
        ref = full.cpu().numpy() if hasattr(full, "cpu") else full
        for i in range(0, streams.size, max(1, streams.size // 200)):
            assert np.array_equal(got[offs[i]:offs[i + 1]], ref[streams[i], first[i]:last[i]]), (name, i)
        frames, fbytes = touched(h_comp, starts, nbytes, streams, first, last)
        out_b = int(offs[-1]) * 4
        med, lo, hi = timed(lambda: far.to_windows(streams, first, last), args.reps)
        emit(dict(case=name, windows=int(streams.size), window_samples=length, residency="device", ms_median=med, ms_min=lo,
                  ms_max=hi, reps=args.reps, frames_touched=frames, touched_frame_bytes=fbytes, output_bytes=out_b,
                  gbs=(fbytes + out_b) / (med * 1e-3) / 1e9))
        if name == "a":
            comp_h, offs_h = h_comp, None
            off, gain = np.asarray(far.stream_offsets).reshape(-1), np.asarray(far.stream_gains).reshape(-1)

            def host_call():
                return fa.array_decompress_windows(comp_h, n, starts, nbytes, streams, first, last, stream_offsets=off,
                                                   stream_gains=gain)

            d_h, offs_h = host_call()
            assert np.array_equal(d_h, got)
            med_h, lo_h, hi_h = timed(host_call, args.reps)
            emit(dict(case="a", windows=int(streams.size), window_samples=length, residency="host", ms_median=med_h,
                      ms_min=lo_h, ms_max=hi_h, reps=args.reps, frames_touched=frames, touched_frame_bytes=fbytes,
                      output_bytes=out_b, gbs=(fbytes + out_b) / (med_h * 1e-3) / 1e9))

            def loop():
                return [far[int(s), int(a):int(b)] for s, a, b in zip(streams, first, last)]

            res = loop()
            assert all(np.array_equal(np.asarray(r.cpu() if hasattr(r, "cpu") else r).reshape(-1),
                                      got[offs[i]:offs[i + 1]]) for i, r in enumerate(res[:50]))
            med_l, lo_l, hi_l = timed(loop, args.loop_reps, warmup=1)
            emit(dict(case="a", variant="far[s, a:b] loop", windows=int(streams.size), ms_median=med_l, ms_min=lo_l,
                      ms_max=hi_l, reps=args.loop_reps))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for d in lines:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
