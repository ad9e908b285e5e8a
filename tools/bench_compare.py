"""Comparisons and is.na() on the C2 shape (33,538 x 1,000,000 integer counts
at density 0.07, nnz = 2.348e9, generated in HBM): CUDA-event times
(median of --reps runs after a warm-up) of

  x > 0          NA rate 1e-6 (the 1 / NA value array is written) and NA
                 rate 0 (nothing dropped: leaf_ptr + offsets copied)
  x > 1          about 3.6 % kept
  x > v          a per-row threshold v[i] = i % 3
  z > t          z = log1p(sweep(x, 2, sf, "/")), t = the median stored
                 value of z (about half kept)
  is.na(x)
  colSums / rowSums of x > 0 (NA rate 0: a lacunar result)

each with the bytes it must move (from nnz and the kept count) and the
fraction of the 6546 GB/s measured copy bandwidth; the host alternative
(numpy filter of the CSC, then from_csc) on the first 100,000 columns; the
card name and power limit from the same run.  Prints one JSON line.

    python tools/bench_compare.py [--ncol N] [--reps R]
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


def has_vals(h):
    import ctypes
    from sparsearray_b200 import _native
    fl = ctypes.c_int(0)
    _native.check(_native.lib().svtgpu_matrix_info(
        h._h, None, None, None, None, ctypes.byref(fl)))
    return bool(fl.value & _native.HAS_VALS)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncol", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-cols", type=int, default=100_000)
    args = ap.parse_args()
    import torch
    import sparsearray_b200 as sa
    from sparsearray_b200 import synth
    from sparsearray_b200.device import DeviceSVT

    ncol = args.ncol
    res = {"device": device_card(), "shape": [NROW, ncol],
           "peak_copy_GBs": PEAK_GBS, "ops": {}}
    keep = {}

    def record(name, fn, bytes_of):
        med, lo, hi = timed(fn, args.reps)
        out = keep.get("r")
        g = bytes_of(out) / 1e9
        row = {"ms": med, "ms_min": lo, "ms_max": hi, "GB": g,
               "GBs": g / med * 1e3, "frac_copy_bw": g / med * 1e3 / PEAK_GBS}
        if out is not None:
            row.update(nnz_out=out.nnz, value_array=has_vals(out))
        res["ops"][name] = row
        keep.pop("r", None)

    lp = 8.0 * (ncol + 1)

    def filt(nnz, x_bytes, offs_in_count):
        """count pass: the values (+ the offsets for a per-row operand);
        then either the copy of the offsets (nothing dropped, no NA) or the
        write pass: offsets + values again, the kept offsets (+ 1 / NA values
        when the result stores them) written; leaf_ptr read and written."""
        def f(out):
            b = nnz * (x_bytes + 4 * offs_in_count)
            if out.nnz == nnz and not has_vals(out):
                b += 8 * nnz
            else:
                b += nnz * (4 + x_bytes) + out.nnz * (4 + 4 * has_vals(out))
            return b + 3 * lp
        return f

    # --- NA rate 0: x > 0 keeps everything, no NA -> copy path ---------
    x0 = DeviceSVT.generate_poisson(NROW, ncol, DENSITY, seed=SEED)
    n0 = x0.nnz
    record("gt0_no_na", lambda: keep.__setitem__(
        "r", x0.ewise(">", np.array([0], np.int32))),
        filt(n0, 4, 0))
    y = x0.ewise(">", np.array([0], np.int32))
    record("colSums_of_gt0_lacunar",
           lambda: y.colstats("sum"), lambda _: 8.0 * ncol + 8.0 * ncol)
    record("rowSums_of_gt0_lacunar",
           lambda: y.rowstats("sum"), lambda _: 4.0 * n0 + lp)
    del y, x0

    # --- NA rate 1e-6 --------------------------------------------------
    x = DeviceSVT.generate_poisson(NROW, ncol, DENSITY, seed=SEED,
                                   na_rate=NA_RATE)
    nnz = x.nnz
    res["nnz"] = nnz
    for name, op, v, margin, off in (
            ("gt0_with_na", ">", np.array([0], np.int32), 0, 0),
            ("gt1", ">", np.array([1], np.int32), 0, 0),
            ("gt_per_row", ">", (np.arange(NROW) % 3).astype(np.int32), 1,
             1)):
        record(name, lambda op=op, v=v, margin=margin: keep.__setitem__(
            "r", x.ewise(op, v, margin=margin)),
            filt(nnz, 4, off))
    record("is_na", lambda: keep.__setitem__("r", x.ewise("is.na")),
           filt(nnz, 4, 0))
    y = x.ewise(">", np.array([0], np.int32))
    record("colSums_of_gt0_with_na", lambda: y.colstats("sum"),
           lambda _: 4.0 * nnz + lp)
    record("rowSums_of_gt0_with_na", lambda: y.rowstats("sum"),
           lambda _: 8.0 * nnz + lp)
    del y

    # --- about half kept: log1p(sweep(x, 2, sf, "/")) > median ---------
    cs = x.colstats("sum", na_rm=True)[0].cpu().numpy()
    sf = cs / cs.mean()
    z = x.ewise("/", sf, margin=2).ewise("log1p")
    p, o, v = synth.poisson_csc(NROW, 2000, DENSITY, seed=SEED,
                                na_rate=NA_RATE)
    cols = np.repeat(np.arange(2000), np.diff(p))
    w = np.log1p(v[v != sa.NA_INTEGER] / sf[cols[v != sa.NA_INTEGER]])
    t = float(np.median(w))
    res["half_threshold"] = t
    record("log1p_sweep_gt_median",
           lambda: keep.__setitem__("r", z.ewise(">", np.array([t]))),
           filt(nnz, 8, 0))
    del z, x

    # --- host alternative: numpy filter of the CSC, then from_csc ------
    hc = min(args.host_cols, ncol)
    p, o, v = synth.poisson_csc(NROW, hc, DENSITY, seed=SEED,
                                na_rate=NA_RATE)
    t0 = time.perf_counter()
    na = v == sa.NA_INTEGER
    kept = (v > 1) | na
    cols = np.repeat(np.arange(hc), np.diff(p))
    pk = np.zeros(hc + 1, dtype=np.int64)
    np.cumsum(np.bincount(cols[kept], minlength=hc), out=pk[1:])
    ok, vk = o[kept], np.where(na[kept], sa.NA_INTEGER, 1).astype(np.int32)
    t1 = time.perf_counter()
    r = sa.from_csc((NROW, hc), pk, vk, ok)      # 1 / NA as integers
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    r.release()
    res["host_alternative_gt1"] = {
        "cols": hc, "filter_ms": (t1 - t0) * 1e3,
        "from_csc_ms": (t2 - t1) * 1e3,
        "device_equivalent_ms": res["ops"]["gt1"]["ms"] * hc / ncol}
    print(json.dumps(res))
    return 0


if __name__ == "__main__":
    sys.exit(main())
