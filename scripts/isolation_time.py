"""Time of the isolated decode and of verify against the plain decode on the configs[1] shape.

    python scripts/isolation_time.py [--streams 1000] [--samples 1000000] [--reps 21] [--out FILE]

float32 (streams, samples) detector timestreams (bench.make_tod_torch), quanta 1e-4, level 5, compressed bytes on the
device.  Three device-level calls on the same bytes, each ending in a device synchronise:
  fab_decode           float32 output (fused restore), as FlacArray.to_array() runs it
  fab_decode_isolated  the same, with per-stream status and the fill kernel
  fab_verify           decode and check every frame, store nothing
After a warm-up the three are called in turn, `reps` rounds, so that drifts of the machine hit all three alike; each gets
median / min / max.  The isolated output is checked bit for bit against the plain one, and both statuses must be zero.
Prints one JSON object per line (and writes them to --out, default profiles/r04_isolation_time.jsonl); the first line
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1000)
    ap.add_argument("--samples", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_isolation_time.jsonl"))
    args = ap.parse_args()

    import torch

    import bench
    import flacarray_b200 as fa
    from flacarray_b200 import libflacarray as lf
    from windows_time import gpu_info

    if not torch.cuda.is_available():
        raise SystemExit("isolation_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    emit(dict(gpu_info(), streams=args.streams, samples=args.samples, dtype="float32", quanta=1e-4, level=5,
              residency="device"))
    ns, n = args.streams, args.samples
    x = bench.make_tod_torch(ns, n, 1, dev)
    far = fa.FlacArray.from_array(x, quanta=np.full(ns, 1e-4, np.float32), level=5)
    del x
    comp = far.compressed
    h_st = np.asarray(far.stream_starts).reshape(-1)
    h_nb = np.asarray(far.stream_nbytes).reshape(-1)
    d_st = torch.from_numpy(h_st).to(dev)
    d_nb = torch.from_numpy(h_nb).to(dev)
    off = lf.to_device(np.asarray(far.stream_offsets).reshape(-1), dev, torch.float32)
    gain = lf.to_device(np.asarray(far.stream_gains).reshape(-1), dev, torch.float32)
    max_nb = int(h_nb.max())
    hint = lf.blocksize_hint(comp, h_st)
    status = torch.empty(ns, dtype=torch.int32, device=dev)

    calls = {
        "fab_decode": lambda: lf.decode_device(comp, d_st, d_nb, ns, n, -1, -1, False, max_nb, hint, off, gain),
        "fab_decode_isolated": lambda: lf.decode_device(comp, d_st, d_nb, ns, n, -1, -1, False, max_nb, hint, off, gain,
                                                        status=status),
        "fab_verify": lambda: lf.verify_device(comp, d_st, d_nb, ns, n, False, max_nb, hint, status),
    }
    ref = calls["fab_decode"]()
    iso = calls["fab_decode_isolated"]()
    same = bool(torch.equal(ref.view(torch.int32), iso.view(torch.int32)))
    st_iso = int(torch.count_nonzero(status))
    del ref, iso
    calls["fab_verify"]()
    st_ver = int(torch.count_nonzero(status))
    if not same or st_iso or st_ver:
        raise SystemExit(f"isolated decode differs ({not same}) or flags streams ({st_iso}, {st_ver})")

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
    comp_bytes = int(h_nb.sum())
    for k, ts in times.items():
        med = float(np.median(ts))
        emit(dict(call=k, ms_median=med, ms_min=float(min(ts)), ms_max=float(max(ts)), reps=args.reps,
                  compressed_bytes=comp_bytes, output_bytes=0 if k == "fab_verify" else ns * n * 4,
                  compressed_gbs=comp_bytes / (med * 1e-3) / 1e9))
    emit(dict(check="isolated output bit-identical to fab_decode, zero status from isolated decode and verify",
              passed=True))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for d in lines:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
