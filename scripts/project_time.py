"""Time of FlacArray.project() on the configs[1] shape, next to stats() and to_array() followed by a torch matmul.

    python scripts/project_time.py [--streams 1000] [--samples 1000000] [--reps 21] [--out FILE]

float32 (streams, samples) detector timestreams (bench.make_tod_torch), quanta 1e-4, level 5.  Three template sets:
  cm        1 template: the common mode from combine()
  legendre  3 templates: Legendre polynomials 0-2 over the range
  lockin    16 templates: 8 sine / cosine pairs
Calls, each ending in a device synchronise, alternated `reps` rounds after a warm-up so that drifts of the machine hit
all of them alike; each gets median / min / max ms:
  project_device_<set>       FlacArray.project() with the compressed bytes on the device
  project_host_legendre      the same FlacArray with the bytes in (pageable) host memory
  stats_device               FlacArray.stats() (bin=None) from device bytes
  to_array_matmul_<set>      FlacArray.to_array() on the device, then V.double() @ T.T
k_project_piece + k_project_fold (one fab_project_rows call) alone are timed with CUDA events over the int32 rows of all
streams (the decoded integers, 4 GB at the default shape) for each set: GB/s over the row and template bytes read, and
FP64 GFLOP/s (2 * rows * samples * templates).  Before timing, every set's result is checked bit for bit against the same
fold done with torch on the device (per 4096-sample piece p = p + T[t, i] * v[i] in ascending i, then the pieces in
order) and against the host-resident call.  One JSON object per line (and --out, default profiles/r10_project_time.jsonl);
the first line names the GPU and its power limit.
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

PIECE = 4096


def torch_fold(v, t):
    """The definition with torch on the device: v [ns, n] float64, t [nt, n] float64 -> [ns, nt]."""
    import torch

    ns, n = v.shape
    nt = t.shape[0]
    npc = -(-n // PIECE)
    vp = torch.zeros((ns, npc * PIECE), dtype=torch.float64, device=v.device)
    vp[:, :n] = v
    tp = torch.zeros((nt, npc * PIECE), dtype=torch.float64, device=v.device)
    tp[:, :n] = t
    vp = vp.view(ns, npc, PIECE)
    tp = tp.view(nt, npc, PIECE)
    acc = torch.zeros((ns, nt, npc), dtype=torch.float64, device=v.device)
    for i in range(min(PIECE, n)):
        acc = acc + tp[None, :, :, i] * vp[:, None, :, i]
    out = torch.zeros((ns, nt), dtype=torch.float64, device=v.device)
    for j in range(npc):
        out = out + acc[:, :, j]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1000)
    ap.add_argument("--samples", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--check-streams", type=int, default=64, help="streams of the torch fold check (it is slow)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_project_time.jsonl"))
    args = ap.parse_args()

    import torch

    import bench
    import flacarray_b200 as fa
    from flacarray_b200 import libflacarray as lf
    from windows_time import gpu_info

    if not torch.cuda.is_available():
        raise SystemExit("project_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    ns, n = args.streams, args.samples
    emit(dict(gpu_info(), streams=ns, samples=n, dtype="float32", quanta=1e-4, level=5, piece=PIECE,
              group_cap_bytes=lf._STATS_GROUP_BYTES))
    x = bench.make_tod_torch(ns, n, 1, dev)
    far = fa.FlacArray.from_array(x, quanta=np.full(ns, 1e-4, np.float32), level=5)
    del x
    far_h = fa.FlacArray(far)
    far_h._compressed = far.compressed.cpu().numpy()
    far_h._init_params()

    s = np.linspace(-1.0, 1.0, n)
    k = np.arange(n)
    sets = {
        "cm": far.combine().view(1, n).contiguous(),
        "legendre": torch.from_numpy(np.stack([np.ones(n), s, 1.5 * s * s - 0.5])).to(dev),
        "lockin": torch.from_numpy(np.stack([f(2 * np.pi * h * k / 1000.0) for h in range(1, 9)
                                             for f in (np.sin, np.cos)])).to(dev),
    }

    # correctness on this data: the torch fold on the device (over the first streams: it loops over 4096 positions),
    # and host residency, give the same bits
    arr = far.to_array()
    m = min(args.check_streams, ns)
    for name, t in sets.items():
        got = far.project(t)
        want = torch_fold(arr[:m].double(), t)
        same_fold = bool(torch.equal(got[:m].view(torch.int64), want.view(torch.int64)))
        same_host = bool(np.array_equal(got.cpu().numpy().view(np.uint8), far_h.project(t.cpu()).view(np.uint8)))
        emit(dict(check=f"project {name}: bits vs the torch fold on the device ({m} streams) and vs host-resident bytes "
                        f"(all streams)", bits_equal_torch_fold=same_fold, bits_equal_host=same_host,
                  templates=int(t.shape[0])))
        if not same_fold or not same_host:
            raise SystemExit(f"project {name} does not match the fold")
        del got, want
    del arr

    def matmul(t):
        return lambda: far.to_array().double() @ t.T

    calls = {}
    for name, t in sets.items():
        calls[f"project_device_{name}"] = (lambda t=t: far.project(t))
    calls["project_host_legendre"] = lambda: far_h.project(sets["legendre"])
    calls["stats_device"] = lambda: far.stats()
    for name, t in sets.items():
        calls[f"to_array_matmul_{name}"] = matmul(t)
    for _ in range(args.warmup):
        for fn in calls.values():
            fn()
    torch.cuda.synchronize()
    times = {k_: [] for k_ in calls}
    for _ in range(args.reps):
        for k_, fn in calls.items():
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            times[k_].append((time.perf_counter() - t0) * 1e3)
            del out
    comp_bytes = int(np.asarray(far.stream_nbytes).sum())
    for k_, ts in times.items():
        med = float(np.median(ts))
        emit(dict(call=k_, ms_median=med, ms_min=float(min(ts)), ms_max=float(max(ts)), reps=args.reps,
                  compressed_bytes=comp_bytes, decoded_gbs=ns * n * 4 / (med * 1e-3) / 1e9))

    # fab_project_rows alone (k_project_piece + k_project_fold) over the int32 rows of every stream
    h_st = np.asarray(far.stream_starts).reshape(-1)
    h_nb = np.asarray(far.stream_nbytes).reshape(-1)
    ints = lf.decode_device(far.compressed, torch.from_numpy(h_st).to(dev), torch.from_numpy(h_nb).to(dev), ns, n, -1, -1,
                            False, int(h_nb.max()), lf.blocksize_hint(far.compressed, h_st))
    off = torch.from_numpy(np.asarray(far.stream_offsets).reshape(-1).copy()).to(dev)
    gain = torch.from_numpy(np.asarray(far.stream_gains).reshape(-1).copy()).to(dev)
    for name, t in sets.items():
        nt = int(t.shape[0])
        out = torch.empty((ns, nt), dtype=torch.float64, device=dev)

        def run():
            lf.project_device(ints, False, ns, n, off, gain, None, t, nt, out)

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
        tmpl_bytes = nt * n * 8
        flop = 2 * ns * n * nt
        emit(dict(kernel=f"fab_project_rows ({name}: k_project_piece + k_project_fold)", templates=nt, rows=ns, samples=n,
                  row_bytes=row_bytes, template_bytes=tmpl_bytes, ms_median=med, ms_min=float(min(ms)),
                  ms_max=float(max(ms)), gbs=(row_bytes + tmpl_bytes) / (med * 1e-3) / 1e9,
                  fp64_gflops=flop / (med * 1e-3) / 1e9))
        del out
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for d in lines:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
