"""`x op y` between two SVTs on the C2 shape (33,538 x 1,000,000 integer
counts at density 0.07, nnz = 2.348e9 each), generated twice in HBM with
seeds A and B: CUDA-event times (median of --reps runs after a warm-up) of

  x + y          int, union about 4.53e9 entries (above 2^32)
  x * y          int, about 164e6 kept
  (x>0) & (y>0)  lacunar inputs (generated without values), lacunar result
  x != y         int
  z1 - z2        double, zk = log1p(sweep(xk, 2, sf_k, "/")), on the first
                 --dcols columns (500,000 by default)

each with the bytes the passes move (count pass: both inputs read; write
pass: both inputs read again and the result written once) next to the
minimum (both inputs read once, the result written once), and the fraction
of the 6546 GB/s measured copy bandwidth on each; the host alternative
(scipy CSC `+`, then from_csc) on the first --host-cols columns; the card
name and power limit from the same run.  Prints one JSON line.

    python tools/bench_ops2.py [--ncol N] [--dcols N] [--reps R]
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NROW, DENSITY, SEED_A, SEED_B, NA_RATE = 33538, 0.07, 2, 3, 1e-6
PEAK_GBS = 6546.0


def device_card():
    try:
        out = subprocess.run(
            ["nvidia-smi", "--query-gpu=name,power.limit",
             "--format=csv,noheader"], capture_output=True, text=True,
            timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:          # the query is informative only
        return "unknown (%s)" % e


def timed(fn, reps):
    import torch
    fn()                                        # warm-up (allocations)
    times = []
    for _ in range(reps):
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(min(times)), float(max(times))


def has_vals(h):
    import ctypes
    from sparsearray_b200 import _native
    fl = ctypes.c_int(0)
    _native.check(_native.lib().svtgpu_matrix_info(
        h._h, None, None, None, None, ctypes.byref(fl)))
    return bool(fl.value & _native.HAS_VALS)


def entry_bytes(d):
    return 4 + (0 if d.vals is None and not has_vals(d) else
                8 if d.val_type == "double" else 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncol", type=int, default=1_000_000)
    ap.add_argument("--dcols", type=int, default=500_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-cols", type=int, default=100_000)
    args = ap.parse_args()
    import torch
    import scipy.sparse as sp
    import sparsearray_b200 as sa
    from sparsearray_b200 import synth
    from sparsearray_b200.device import DeviceSVT

    ncol = args.ncol
    res = {"device": device_card(), "shape": [NROW, ncol],
           "peak_copy_GBs": PEAK_GBS, "ops": {}}
    keep = {}

    def record(name, fn, x, y):
        med, lo, hi = timed(fn, args.reps)
        out = keep.pop("r")
        lp = 8.0 * (x.nleaf + 1)
        read = x.nnz * entry_bytes(x) + y.nnz * entry_bytes(y) + 2 * lp
        write = out.nnz * entry_bytes(out) + lp
        g_min, g = (read + write) / 1e9, (2 * read + write) / 1e9
        res["ops"][name] = {
            "ms": med, "ms_min": lo, "ms_max": hi, "nnz_out": out.nnz,
            "value_array": has_vals(out), "GB_moved": g, "GB_min": g_min,
            "floor_ms": g_min / PEAK_GBS * 1e3,
            "frac_copy_bw_moved": g / med * 1e3 / PEAK_GBS,
            "frac_copy_bw_min": g_min / med * 1e3 / PEAK_GBS,
            "warnings": out.warnings}
        del out
        gc.collect()

    def run(x, op, y):
        return lambda: keep.__setitem__("r", x.ewise_svt(op, y))

    x = DeviceSVT.generate_poisson(NROW, ncol, DENSITY, seed=SEED_A,
                                   na_rate=NA_RATE)
    y = DeviceSVT.generate_poisson(NROW, ncol, DENSITY, seed=SEED_B,
                                   na_rate=NA_RATE)
    res["nnz"] = [x.nnz, y.nnz]
    for name, op in (("add_int", "+"), ("mul_int", "*"), ("ne_int", "!=")):
        record(name, run(x, op, y), x, y)
    del x, y
    gc.collect()

    xl = DeviceSVT.generate_poisson(NROW, ncol, DENSITY, seed=SEED_A,
                                    lacunar=True)
    yl = DeviceSVT.generate_poisson(NROW, ncol, DENSITY, seed=SEED_B,
                                    lacunar=True)
    record("and_lacunar", run(xl, "&", yl), xl, yl)
    del xl, yl
    gc.collect()

    dc = min(args.dcols, ncol)
    zs = []
    for seed in (SEED_A, SEED_B):
        x = DeviceSVT.generate_poisson(NROW, dc, DENSITY, seed=seed,
                                       na_rate=NA_RATE)
        cs = x.colstats("sum", na_rm=True)[0].cpu().numpy()
        zs.append(x.ewise("/", cs / cs.mean(), margin=2).ewise("log1p"))
        del x
        gc.collect()
    record("sub_double_%dcols" % dc, run(zs[0], "-", zs[1]), zs[0], zs[1])
    del zs
    gc.collect()
    torch.cuda.synchronize()

    # --- host alternative: scipy CSC `+`, then from_csc -----------------
    hc = min(args.host_cols, ncol)
    m = []
    for seed in (SEED_A, SEED_B):
        p, o, v = synth.poisson_csc(NROW, hc, DENSITY, seed=seed)
        m.append(sp.csc_matrix((v, o, p), shape=(NROW, hc)))
    t0 = time.perf_counter()
    s = (m[0] + m[1]).tocsc()
    s.sort_indices()
    t1 = time.perf_counter()
    r = sa.from_csc((NROW, hc), s.indptr, s.data, s.indices)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    r.release()
    res["host_alternative_add"] = {
        "cols": hc, "NA_rate": 0.0, "scipy_add_ms": (t1 - t0) * 1e3,
        "from_csc_ms": (t2 - t1) * 1e3,
        "device_equivalent_ms": res["ops"]["add_int"]["ms"] * hc / ncol}
    print(json.dumps(res))
    return 0


if __name__ == "__main__":
    sys.exit(main())
