"""Time of FlacArray.stats() on the configs[1] shape, next to verify() and to_array() followed by torch reductions.

    python scripts/stats_time.py [--streams 1000] [--samples 1000000] [--reps 21] [--out FILE]

float32 (streams, samples) detector timestreams (bench.make_tod_torch), quanta 1e-4, level 5.  Calls, each ending in a
device synchronise, alternated `reps` rounds after a warm-up so that drifts of the machine hit all of them alike; each
gets median / min / max ms:
  stats_device_bin_none / _bin_4096   FlacArray.stats() with the compressed bytes on the device
  stats_host_bin_none / _bin_4096     the same FlacArray with the bytes in (pageable) host memory
  verify_device                       FlacArray.verify(): decode and check every frame, store nothing
  to_array_torch_device               FlacArray.to_array() on the device, then torch aminmax / mean / std per stream
  stats_device_cap_<MiB>              stats(bin=None) from device bytes with other group caps (how the cap was chosen)
k_row_stats alone is timed with CUDA events over the int32 rows of the first group (the decoded integers of
_STATS_GROUP_BYTES): GB/s over the decoded bytes it reads, and the fraction of 6550 GB/s (the HBM read rate measured
for this project on the B200).  The stats are checked against the decoded array (count, min, max exact; mean and std
close to torch's float64).  One JSON object per line (and --out, default profiles/r06_stats_time.jsonl); the first line
names the GPU and its power limit.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

HBM_GBS = 6550.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1000)
    ap.add_argument("--samples", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_stats_time.jsonl"))
    args = ap.parse_args()

    import torch

    import bench
    import flacarray_b200 as fa
    from flacarray_b200 import libflacarray as lf
    from windows_time import gpu_info

    if not torch.cuda.is_available():
        raise SystemExit("stats_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    ns, n = args.streams, args.samples
    emit(dict(gpu_info(), streams=ns, samples=n, dtype="float32", quanta=1e-4, level=5,
              group_cap_bytes=lf._STATS_GROUP_BYTES))
    x = bench.make_tod_torch(ns, n, 1, dev)
    far = fa.FlacArray.from_array(x, quanta=np.full(ns, 1e-4, np.float32), level=5)
    del x
    far_h = fa.FlacArray(far)
    far_h._compressed = far.compressed.cpu().numpy()
    far_h._init_params()

    # correctness on this data: exact count / min / max, mean / std against torch float64 on the decoded array
    s = far.stats()
    arr = far.to_array()
    mn, mx = torch.aminmax(arr, dim=1)
    a64 = arr.double()
    ok = (np.array_equal(s.min, mn.cpu().numpy()) and np.array_equal(s.max, mx.cpu().numpy())
          and bool((s.count == n).all()))
    d_mean = float(np.abs(s.mean - a64.mean(dim=1).cpu().numpy()).max())
    d_std = float(np.abs(s.std - a64.std(dim=1, correction=0).cpu().numpy()).max())
    amax = float(a64.abs().max())
    del arr, a64, mn, mx
    same_host = all(np.array_equal(u.view(np.uint8), v.view(np.uint8)) for u, v in zip(s, far_h.stats()))
    emit(dict(check="stats vs decoded array: count/min/max exact, mean/std max abs diff vs torch float64",
              exact=bool(ok), mean_max_abs_diff=d_mean, std_max_abs_diff=d_std, max_abs_sample=amax,
              host_bits_equal_device=bool(same_host)))
    if not ok or not same_host:
        raise SystemExit("stats do not match the decoded array")

    def torch_reduce():
        a = far.to_array()
        r = torch.aminmax(a, dim=1), a.mean(dim=1, dtype=torch.float64), a.double().std(dim=1, correction=0)
        return r

    def with_cap(cap):
        def f():
            old = lf._STATS_GROUP_BYTES
            lf._STATS_GROUP_BYTES = cap
            try:
                return far.stats()
            finally:
                lf._STATS_GROUP_BYTES = old
        return f

    calls = {
        "stats_device_bin_none": lambda: far.stats(),
        "stats_device_bin_4096": lambda: far.stats(bin=4096),
        "stats_host_bin_none": lambda: far_h.stats(),
        "stats_host_bin_4096": lambda: far_h.stats(bin=4096),
        "verify_device": lambda: far.verify(),
        "to_array_torch_device": torch_reduce,
    }
    for mib in (256, 1024, 2048, 8192):
        calls[f"stats_device_cap_{mib}"] = with_cap(mib << 20)
    for _ in range(args.warmup):
        for fn in calls.values():
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
    for _ in range(args.reps):
        for k, fn in calls.items():
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            times[k].append((time.perf_counter() - t0) * 1e3)
            del out
    comp_bytes = int(np.asarray(far.stream_nbytes).sum())
    for k, ts in times.items():
        med = float(np.median(ts))
        emit(dict(call=k, ms_median=med, ms_min=float(min(ts)), ms_max=float(max(ts)), reps=args.reps,
                  compressed_bytes=comp_bytes, decoded_gbs=ns * n * 4 / (med * 1e-3) / 1e9))

    # k_row_stats alone over the rows of one group
    rows_per_group = max(1, lf._STATS_GROUP_BYTES // (n * 4))
    g = min(ns, rows_per_group)
    h_st = np.asarray(far.stream_starts).reshape(-1)[:g]
    h_nb = np.asarray(far.stream_nbytes).reshape(-1)[:g]
    ints = lf.decode_device(far.compressed, torch.from_numpy(h_st).to(dev), torch.from_numpy(h_nb).to(dev), g, n, -1, -1,
                            False, int(h_nb.max()), lf.blocksize_hint(far.compressed, h_st))
    off = torch.from_numpy(np.asarray(far.stream_offsets).reshape(-1)[:g].copy()).to(dev)
    gain = torch.from_numpy(np.asarray(far.stream_gains).reshape(-1)[:g].copy()).to(dev)
    for bin_ in (0, 4096):
        nb = 1 if bin_ == 0 else -(-n // bin_)
        res = [torch.empty(g * nb, dtype=t, device=dev)
               for t in (torch.int64, torch.float32, torch.float32, torch.float64, torch.float64)]

        def run():
            lf.row_stats_device(ints, False, g, n, bin_, off, gain, None, *res)

        for _ in range(3):
            run()
        ms = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run()
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        med = float(np.median(ms))
        gbs = g * n * 4 / (med * 1e-3) / 1e9
        emit(dict(kernel="k_row_stats" + ("" if bin_ == 0 else " (bin 4096)"), bin=bin_ or None, rows=g, samples=n,
                  decoded_bytes=g * n * 4, ms_median=med, ms_min=float(min(ms)), ms_max=float(max(ms)), gbs=gbs,
                  fraction_of_6550_gbs=gbs / HBM_GBS))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for d in lines:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
