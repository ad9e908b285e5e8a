"""`x[i, j]` on the C2 shape (33,538 x 1,000,000 integer counts at density
0.07, nnz = 2.348e9), generated in HBM: CUDA-event times around the whole
call (median of --reps runs after a warm-up) of

  cols_90pct      x[, keep], about 90 % of the columns (gather route)
  rows_hvg_sorted x[hvg, ], 2,000 rows in ascending order (row-map route)
  rows_hvg_varord the same rows in decreasing-variance order (unsorted route)
  genes_cells     x[genes, cells], 15,000 sorted rows x 900,000 columns
  cols_lacunar    x[, keep] of the matrix generated without values
  cols_double     x[, keep] of the matrix generated as doubles

each with the bytes its passes move next to the minimum traffic (the
offsets of the selected leaves read once, the values of the kept entries
read once, the result written once), both computed from shapes here, and
the fraction of the 6,546 GB/s measured copy bandwidth on each; the host
alternative (scipy CSC slicing, then from_csc) on the first --host-cols
columns; the card name and power limit from the same run.  Prints one JSON
line.

    python tools/bench_subset.py [--ncol N] [--reps R] [--host-cols N]
"""
import argparse
import ctypes
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NROW, DENSITY, SEED, NA_RATE = 33538, 0.07, 2, 1e-6
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


def has_vals(d):
    from sparsearray_b200 import _native
    fl = ctypes.c_int(0)
    _native.check(_native.lib().svtgpu_matrix_info(
        d._h, None, None, None, None, ctypes.byref(fl)))
    return bool(fl.value & _native.HAS_VALS)


def leaf_ptr(d):
    from sparsearray_b200 import _native
    p = np.zeros(d.nleaf + 1, np.int64)
    _native.check(_native.lib().svtgpu_matrix_download(
        d._h, p.ctypes.data_as(ctypes.c_void_p), None, None))
    return p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncol", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-cols", type=int, default=100_000)
    args = ap.parse_args()
    import torch
    import scipy.sparse as sp
    import sparsearray_b200 as sa
    from sparsearray_b200 import synth
    from sparsearray_b200.device import DeviceSVT

    ncol = args.ncol
    rng = np.random.Generator(np.random.PCG64(1))
    keep = np.flatnonzero(rng.random(ncol) < 0.9)
    hvg = np.sort(rng.choice(NROW, 2000, replace=False))
    genes = np.sort(rng.choice(NROW, 15000, replace=False))
    cells = np.sort(rng.choice(ncol, ncol * 9 // 10, replace=False))
    res = {"device": device_card(), "shape": [NROW, ncol],
           "peak_copy_GBs": PEAK_GBS, "ops": {}}

    def record(name, x, rows, leaves, route):
        xp = leaf_ptr(x)
        out = {}
        med, lo, hi = timed(lambda: out.__setitem__(
            "r", x.subset(rows, leaves)), args.reps)
        r = out.pop("r")
        vs = (8 if x.val_type == "double" else 4) if has_vals(x) else 0
        eb = 4 + vs
        lens = np.diff(xp) if leaves is None else np.diff(xp)[leaves]
        t_in = float(lens.sum())                # gathered entries
        n_out = float(r.nnz)
        lp = 8.0 * (r.nleaf + 1)
        if route == "gather":
            g_min = 2 * eb * n_out + lp
            g = g_min + 2 * lp                  # lengths, scan, leaf_ptr
        else:
            g_min = 4 * t_in + vs * n_out + eb * n_out + lp
            g = 4 * t_in + g_min                # count pass reads offsets
            if route == "unsorted":             # two transposes (count,
                g += 2 * (4 * n_out + 2 * eb * n_out)   # write) and a
                g += 2 * eb * n_out                     # gather
        g_min, g = g_min / 1e9, g / 1e9
        res["ops"][name] = {
            "route": route, "ms": med, "ms_min": lo, "ms_max": hi,
            "nnz_in_gathered": int(t_in), "nnz_out": int(n_out),
            "value_array": has_vals(r), "GB_moved": g, "GB_min": g_min,
            "floor_ms": g_min / PEAK_GBS * 1e3,
            "frac_copy_bw_moved": g / med * 1e3 / PEAK_GBS,
            "frac_copy_bw_min": g_min / med * 1e3 / PEAK_GBS}
        del r
        gc.collect()

    x = DeviceSVT.generate_poisson(NROW, ncol, DENSITY, seed=SEED,
                                   na_rate=NA_RATE)
    res["nnz"] = x.nnz
    record("cols_90pct", x, None, keep, "gather")
    record("rows_hvg_sorted", x, hvg, None, "rowmap")
    # the same rows by decreasing rowVars (not part of the timing)
    var = x.rowmoments(na_rm=True)[1].cpu().numpy()
    order = hvg[np.argsort(-var[hvg], kind="stable")]
    record("rows_hvg_varord", x, order, None, "unsorted")
    record("genes_cells", x, genes, cells, "rowmap")
    del x
    gc.collect()
    xl = DeviceSVT.generate_poisson(NROW, ncol, DENSITY, seed=SEED,
                                    lacunar=True)
    record("cols_lacunar", xl, None, keep, "gather")
    del xl
    gc.collect()
    xd = DeviceSVT.generate_poisson(NROW, ncol, DENSITY, seed=SEED,
                                    na_rate=NA_RATE, val_type="double")
    record("cols_double", xd, None, keep, "gather")
    del xd
    gc.collect()
    torch.cuda.synchronize()

    # --- host alternative: scipy CSC slicing, then from_csc -------------
    hc = min(args.host_cols, ncol)
    p, o, v = synth.poisson_csc(NROW, hc, DENSITY, seed=SEED)
    m = sp.csc_matrix((v, o, p), shape=(NROW, hc))
    hk = keep[keep < hc]
    host = {"cols": hc}
    for name, fn in (("cols_90pct", lambda: m[:, hk]),
                     ("rows_hvg_sorted", lambda: m[hvg, :])):
        t0 = time.perf_counter()
        s = fn().tocsc()
        s.sort_indices()
        t1 = time.perf_counter()
        r = sa.from_csc(s.shape, s.indptr, s.data, s.indices)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        r.release()
        host[name] = {"scipy_ms": (t1 - t0) * 1e3,
                      "from_csc_ms": (t2 - t1) * 1e3,
                      "device_equivalent_ms":
                          res["ops"][name]["ms"] * hc / ncol}
    res["host_alternative"] = host
    print(json.dumps(res))
    return 0


if __name__ == "__main__":
    sys.exit(main())
