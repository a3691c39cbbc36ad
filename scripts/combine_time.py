"""Time of FlacArray.combine() on the configs[1] shape, next to stats() and to_array() followed by torch reductions.

    python scripts/combine_time.py [--streams 1000] [--samples 1000000] [--reps 21] [--out FILE]

float32 (streams, samples) detector timestreams (bench.make_tod_torch), quanta 1e-4, level 5.  Three groupings:
  common   groups=None: the common mode of all streams
  groups7  groups = stream index % 7, weights 1: seven interleaved groups (host staging gathers their bytes)
  pairs    groups = stream index // 2, weights +1 / -1: streams / 2 pair differences
Calls, each ending in a device synchronise, alternated `reps` rounds after a warm-up so that drifts of the machine hit
all of them alike; each gets median / min / max ms:
  combine_device_<grouping>           FlacArray.combine() with the compressed bytes on the device
  combine_host_<grouping>             the same FlacArray with the bytes in (pageable) host memory
  stats_device                        FlacArray.stats() (bin=None) from device bytes
  to_array_torch_<grouping>           FlacArray.to_array() on the device, then the torch reduction of the grouping
k_combine_rows alone is timed with CUDA events over the int32 rows of all streams (the decoded integers, 4 GB at the
default shape) for each grouping: GB/s over the row bytes it reads, and over the row bytes plus the output it reads and
writes.  Before timing, every grouping's result is checked bit for bit against the same fold done with torch on the
device (acc = acc + w * x.double(), one elementwise multiply and add per stream) and against the host-resident call.
One JSON object per line (and --out, default profiles/r07_combine_time.jsonl); the first line names the GPU and its power
limit.
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_combine_time.jsonl"))
    args = ap.parse_args()

    import torch

    import bench
    import flacarray_b200 as fa
    from flacarray_b200 import libflacarray as lf
    from windows_time import gpu_info

    if not torch.cuda.is_available():
        raise SystemExit("combine_time.py needs a CUDA device")
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

    idx = np.arange(ns)
    groupings = {
        "common": (None, None),
        "groups7": (None, idx % 7),
        "pairs": (np.where(idx % 2 == 0, 1.0, -1.0), idx // 2),
    }

    # correctness on this data: the torch fold on the device, and host residency, give the same bits
    arr = far.to_array()
    for name, (w, g) in groupings.items():
        got = far.combine(weights=w, groups=g)
        wt = torch.ones(ns, dtype=torch.float64, device=dev) if w is None else torch.from_numpy(w).to(dev)
        gg = np.zeros(ns, np.int64) if g is None else g
        n_out = int(gg.max()) + 1
        acc = torch.zeros((n_out, n), dtype=torch.float64, device=dev)
        members = [np.flatnonzero(gg == k) for k in range(n_out)]
        for step in range(max(len(m) for m in members)):
            rows = [k for k in range(n_out) if step < len(members[k])]
            src = torch.from_numpy(np.array([members[k][step] for k in rows])).to(dev)
            dst = torch.from_numpy(np.array(rows)).to(dev)
            acc[dst] = acc[dst] + wt[src, None] * arr[src].double()
        want = acc[0] if g is None else acc
        same_fold = bool(torch.equal(got.view(torch.int64), want.view(torch.int64)))
        same_host = bool(np.array_equal(got.cpu().numpy().view(np.uint8), far_h.combine(weights=w, groups=g).view(np.uint8)))
        emit(dict(check=f"combine {name}: bits vs the torch fold on the device and vs host-resident bytes",
                  bits_equal_torch_fold=same_fold, bits_equal_host=same_host, out_rows=n_out))
        if not same_fold or not same_host:
            raise SystemExit(f"combine {name} does not match the fold")
        del acc, got, want
    del arr

    gt7 = torch.from_numpy(idx % 7).to(dev)

    def torch_common():
        return far.to_array().sum(dim=0, dtype=torch.float64)

    def torch_groups7():
        a = far.to_array()
        return torch.zeros((7, n), dtype=torch.float64, device=dev).index_add_(0, gt7, a.double())

    def torch_pairs():
        a = far.to_array()
        return a[0::2].double() - a[1::2].double()

    calls = {}
    for name, (w, g) in groupings.items():
        calls[f"combine_device_{name}"] = (lambda w=w, g=g: far.combine(weights=w, groups=g))
    for name, (w, g) in groupings.items():
        calls[f"combine_host_{name}"] = (lambda w=w, g=g: far_h.combine(weights=w, groups=g))
    calls["stats_device"] = lambda: far.stats()
    calls["to_array_torch_common"] = torch_common
    calls["to_array_torch_groups7"] = torch_groups7
    calls["to_array_torch_pairs"] = torch_pairs
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

    # k_combine_rows alone over the int32 rows of every stream
    h_st = np.asarray(far.stream_starts).reshape(-1)
    h_nb = np.asarray(far.stream_nbytes).reshape(-1)
    ints = lf.decode_device(far.compressed, torch.from_numpy(h_st).to(dev), torch.from_numpy(h_nb).to(dev), ns, n, -1, -1,
                            False, int(h_nb.max()), lf.blocksize_hint(far.compressed, h_st))
    off = torch.from_numpy(np.asarray(far.stream_offsets).reshape(-1).copy()).to(dev)
    gain = torch.from_numpy(np.asarray(far.stream_gains).reshape(-1).copy()).to(dev)
    for name, (w, g) in groupings.items():
        gg = np.zeros(ns, np.int64) if g is None else g
        order = np.argsort(gg, kind="stable")
        bounds, outs, _ = lf._segments(gg[order], [(0, ns)])
        n_out = int(gg.max()) + 1
        rows = ints if np.array_equal(order, idx) else ints.view(ns, n)[torch.from_numpy(order).to(dev)]
        wt = torch.from_numpy(np.ones(ns) if w is None else w[order]).to(dev)
        d_b = torch.from_numpy(bounds).to(dev)
        d_o = torch.from_numpy(outs).to(dev)
        out = torch.zeros((n_out, n), dtype=torch.float64, device=dev)

        def run():
            lf.combine_device(rows, False, ns, n, off, gain, None, wt, d_b, d_o, outs.size, out, n_out)

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
        row_bytes = ns * n * 4
        out_bytes = 2 * n_out * n * 8
        emit(dict(kernel=f"k_combine_rows ({name})", segments=int(outs.size), rows=ns, samples=n, row_bytes=row_bytes,
                  out_read_write_bytes=out_bytes, ms_median=med, ms_min=float(min(ms)), ms_max=float(max(ms)),
                  row_gbs=row_bytes / (med * 1e-3) / 1e9, total_gbs=(row_bytes + out_bytes) / (med * 1e-3) / 1e9))
        del rows, out
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for d in lines:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
