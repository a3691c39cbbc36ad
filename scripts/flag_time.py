"""Time of FlacArray.flag_ranges() on the configs[1] shape, next to stats() and to_array() followed by a torch mask and
run finding.

    python scripts/flag_time.py [--streams 1000] [--samples 1000000] [--reps 21] [--out FILE]

float32 (streams, samples) detector timestreams (bench.make_tod_torch), quanta 1e-4, level 5, pad 0.  Two threshold sets,
per stream from stats():
  sparse   lo / hi = mean -+ 6 std: the glitch search, few flagged samples
  dense    hi = mean alone: about half of the samples flagged in short runs, the worst case for the number of ranges
           (checked against the host-resident call for the sparse set only, to bound host memory)
Calls, each ending in a device synchronise, alternated `reps` rounds after a warm-up so that drifts of the machine hit
all of them alike; each gets median / min / max ms:
  flags_device_<set>        FlacArray.flag_ranges() with the compressed bytes on the device
  flags_host_sparse         the same FlacArray with the bytes in (pageable) host memory
  stats_device              FlacArray.stats() (bin=None) from device bytes
  to_array_torch_<set>      FlacArray.to_array() on the device, then the torch mask, run starts / ends found with
                            nonzero on the mask's differences, and the ranges copied to the host
The passes alone are timed with CUDA events over the int32 rows of all streams (the decoded integers, 4 GB at the default
shape): fab_flag_count (scan + offsets) and fab_flag_write, next to fab_row_stats over the same rows; GB/s over the row
bytes.  Before timing, both sets are checked against the torch runs and against the host-resident call.  One JSON object
per line (and --out, default profiles/r09_flags_time.jsonl); the first line names the GPU and its power limit.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1000)
    ap.add_argument("--samples", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_flags_time.jsonl"))
    args = ap.parse_args()

    import torch

    import bench
    import flacarray_b200 as fa
    from flacarray_b200 import _lib
    from flacarray_b200 import libflacarray as lf
    from windows_time import gpu_info

    if not torch.cuda.is_available():
        raise SystemExit("flag_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    ns, n = args.streams, args.samples
    emit(dict(gpu_info(), streams=ns, samples=n, dtype="float32", quanta=1e-4, level=5, pad=0,
              group_cap_bytes=lf._STATS_GROUP_BYTES))
    x = bench.make_tod_torch(ns, n, 1, dev)
    far = fa.FlacArray.from_array(x, quanta=np.full(ns, 1e-4, np.float32), level=5)
    del x
    far_h = fa.FlacArray(far)
    far_h._compressed = far.compressed.cpu().numpy()
    far_h._init_params()
    s = far.stats()
    sets = {"sparse": (s.mean - 6 * s.std, s.mean + 6 * s.std), "dense": (None, s.mean)}

    def torch_runs(lo, hi):
        a = far.to_array()
        m = torch.zeros((ns, n + 2), dtype=torch.int8, device=dev)
        mk = torch.zeros((ns, n), dtype=torch.bool, device=dev)
        if lo is not None:
            mk |= a.double() < torch.from_numpy(lo).to(dev)[:, None]
        if hi is not None:
            mk |= a.double() > torch.from_numpy(hi).to(dev)[:, None]
        m[:, 1:-1] = mk.to(torch.int8)
        d = m[:, 1:] - m[:, :-1]
        st = torch.nonzero(d == 1)
        en = torch.nonzero(d == -1)
        return st[:, 0].cpu().numpy(), st[:, 1].cpu().numpy(), en[:, 1].cpu().numpy()

    for name, (lo, hi) in sets.items():
        r = far.flag_ranges(lo=lo, hi=hi)
        ts, tf, tl = torch_runs(lo, hi)
        same_torch = bool(np.array_equal(r.stream, ts) and np.array_equal(r.first, tf) and np.array_equal(r.last, tl))
        rh = far_h.flag_ranges(lo=lo, hi=hi) if name == "sparse" else r       # (dense: host memory for one copy)
        same_host = all(np.array_equal(a, b) for a, b in zip(r, rh))
        emit(dict(check=f"flag_ranges {name}: ranges vs torch runs on to_array() and vs host-resident bytes",
                  equal_torch=same_torch, equal_host=same_host, ranges=int(r.stream.size),
                  flagged=int(r.nflagged.sum())))
        if not same_torch or not same_host:
            raise SystemExit(f"flag_ranges {name} does not match")
        del r, rh

    calls = {}
    for name, (lo, hi) in sets.items():
        calls[f"flags_device_{name}"] = (lambda lo=lo, hi=hi: far.flag_ranges(lo=lo, hi=hi))
    calls["flags_host_sparse"] = lambda: far_h.flag_ranges(lo=sets["sparse"][0], hi=sets["sparse"][1])
    calls["stats_device"] = lambda: far.stats()
    for name, (lo, hi) in sets.items():
        calls[f"to_array_torch_{name}"] = (lambda lo=lo, hi=hi: torch_runs(lo, hi))
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

    # the passes alone over the int32 rows of every stream, next to fab_row_stats
    h_st = np.asarray(far.stream_starts).reshape(-1)
    h_nb = np.asarray(far.stream_nbytes).reshape(-1)
    ints = lf.decode_device(far.compressed, torch.from_numpy(h_st).to(dev), torch.from_numpy(h_nb).to(dev), ns, n, -1, -1,
                            False, int(h_nb.max()), lf.blocksize_hint(far.compressed, h_st))
    off = torch.from_numpy(np.asarray(far.stream_offsets).reshape(-1).copy()).to(dev)
    gain = torch.from_numpy(np.asarray(far.stream_gains).reshape(-1).copy()).to(dev)
    ws = int(_lib.lib().fab_flag_ranges_workspace_bytes(ns, n, 0))
    work = torch.empty(ws, dtype=torch.uint8, device=dev)
    cnt = torch.empty(2 * ns, dtype=torch.int64, device=dev)
    res = [torch.empty(ns, dtype=torch.int64, device=dev) for _ in range(3)] + \
        [torch.empty(ns, dtype=torch.float32, device=dev) for _ in range(2)]
    res += [torch.empty(ns, dtype=torch.float64, device=dev) for _ in range(2)]

    def timed(run):
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
        return float(np.median(ms)), float(min(ms)), float(max(ms))

    row_bytes = ns * n * 4
    for name, (lo, hi) in sets.items():
        d_lo = torch.from_numpy(np.full(ns, -np.inf) if lo is None else lo).to(dev)
        d_hi = torch.from_numpy(hi).to(dev)

        def count():
            lf.flag_count_device(ints, False, ns, n, d_lo, d_hi, off, gain, None, 0, work, cnt[:ns], cnt[ns:])

        med, mn, mx = timed(count)
        emit(dict(kernel=f"fab_flag_count ({name}: k_flag_scan + k_flag_offsets)", rows=ns, samples=n,
                  row_bytes=row_bytes, mask_bytes=ns * ((n + 34) // 32) * 4, ms_median=med, ms_min=mn, ms_max=mx,
                  row_gbs=row_bytes / (med * 1e-3) / 1e9))
        nr = cnt[ns:].cpu().numpy()
        m = int(nr.sum())
        if m == 0:                                      # flag_ranges does not call fab_flag_write without ranges either
            emit(dict(kernel=f"fab_flag_write ({name}: k_flag_write)", ranges=0, note="no ranges: not called"))
            continue
        base = torch.from_numpy(np.concatenate([[0], np.cumsum(nr)[:-1]]).astype(np.int64)).to(dev)
        out = torch.empty(2 * max(m, 1), dtype=torch.int64, device=dev)

        def write():
            lf.flag_write_device(ints, False, ns, n, None, 0, work, base, 0, out[:m], out[m:2 * m])

        med, mn, mx = timed(write)
        emit(dict(kernel=f"fab_flag_write ({name}: k_flag_write)", rows=ns, samples=n, ranges=m,
                  out_bytes=16 * m, ms_median=med, ms_min=mn, ms_max=mx))
        del out

    def stats():
        lf.row_stats_device(ints, False, ns, n, 0, off, gain, None, res[0], res[3], res[4], res[5], res[6])

    med, mn, mx = timed(stats)
    emit(dict(kernel="fab_row_stats (k_row_stats, bin=None)", rows=ns, samples=n, row_bytes=row_bytes, ms_median=med,
              ms_min=mn, ms_max=mx, row_gbs=row_bytes / (med * 1e-3) / 1e9))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for d in lines:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
