"""colMedians() / rowMedians() on matrices generated in HBM: CUDA-event times
(median of --reps runs after a warm-up) of

  1. C2 (33,538 x 1e6 integer counts, d = 0.07, NA rate 1e-6):
     colMedians(na.rm = TRUE) beside colSums of the same arrays through the
     wide kernel (a fresh handle per run, so no compact copy is used)
  2. C2 rowMedians, the device transpose build timed on its own
  3. 33,538 x 110,000 at d = 0.6 (2.2e9 nonzeros, every column selects):
     colMedians and rowMedians
  4. log1p(sweep(x, 2, sf, "/")) of matrix 3: colMedians on double keys

each with the work-list length, the bytes read by classify (values +
leaf_ptr) plus selection (the values its passes read, counted by the kernel)
and those bytes as a share of the 6,546 GB/s measured copy bandwidth; the
card name and power limit from the same run.  Prints a table and one JSON
line.

    python tools/bench_medians.py [--reps R] [--ncol-c2 N] [--ncol-d6 N]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NROW = 33538
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


def timed(fn, reps, setup=None):
    """median / min / max ms of fn() between two CUDA events; setup() runs
    before each run, outside the timed window"""
    import torch
    if setup is not None:
        setup()
    fn()                                        # warm-up
    times = []
    for _ in range(reps):
        if setup is not None:
            setup()
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(min(times)), float(max(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ncol-c2", type=int, default=1_000_000)
    ap.add_argument("--ncol-d6", type=int, default=110_000)
    args = ap.parse_args()
    import torch
    from sparsearray_b200 import _native as N
    from sparsearray_b200.device import DeviceSVT
    if N.device_count() < 1:
        raise SystemExit("bench_medians.py: no CUDA device")
    L = N.lib()
    res = {"device": device_card(), "peak_copy_GBs": PEAK_GBS,
           "reps": args.reps, "ops": {}}

    def selection(h, fn):
        """work-list length and values read by selection, from one
        host-result call on the handle h"""
        fn()
        n, r = ctypes.c_int64(0), ctypes.c_int64(0)
        N.check(L.svtgpu_colmedians_selected(h, ctypes.byref(n),
                                             ctypes.byref(r)))
        return n.value, r.value

    def record(name, ms, bytes_read, **kw):
        row = {"ms": ms[0], "ms_min": ms[1], "ms_max": ms[2]}
        if bytes_read is not None:
            row.update(GB=bytes_read / 1e9,
                       frac_copy_bw=bytes_read / (ms[0] * 1e-3) / 1e9 /
                       PEAK_GBS)
        row.update(kw)
        res["ops"][name] = row
        print("%-28s %9.3f ms  %s" % (name, ms[0], json.dumps(
            {k: v for k, v in row.items() if k not in ("ms",)})),
            flush=True)

    def medians_host(h, nleaf, rows=False):
        out = np.zeros(nleaf)
        fn = L.svtgpu_rowmedians if rows else L.svtgpu_colmedians
        return lambda: N.check(fn(h, 1, out.ctypes.data_as(ctypes.c_void_p)))

    def transpose_ms(x):
        """the device transpose of a fresh handle on x's arrays, events"""
        hs = []

        def setup():
            while hs:                    # its transpose is freed with it
                hs.pop().free()
            hs.append(DeviceSVT(x.nrow, x.nleaf, x.nnz, x.val_type,
                                x.leaf_ptr, x.offs, x.vals))

        def run():
            t = ctypes.c_void_p()
            N.check(L.svtgpu_matrix_transposed(hs[-1]._h, ctypes.byref(t)))
        ms = timed(run, args.reps, setup)
        while hs:
            hs.pop().free()
        return ms

    def medians_workloads(tag, x, vbytes, with_rows):
        lp = 8.0 * (x.nleaf + 1)
        cls_bytes = x.nnz * vbytes + lp
        ms = timed(lambda: x.colmedians(na_rm=True), args.reps)
        n, reads = selection(x._h, medians_host(x._h, x.nleaf))
        record(tag + " colMedians", ms, cls_bytes + reads * vbytes,
               worklist=n, select_values_read=reads)
        if not with_rows:
            return
        record(tag + " transpose build", transpose_ms(x), None)
        rows = medians_host(x._h, x.nrow, rows=True)
        rows()                                   # builds and caches t(x)
        ms = timed(rows, args.reps)
        n, reads = selection(x._h, rows)
        record(tag + " rowMedians", ms,
               x.nnz * vbytes + 8.0 * (x.nrow + 1) + reads * vbytes,
               worklist=n, select_values_read=reads)

    # --- 1, 2: C2 ------------------------------------------------------
    x = DeviceSVT.generate_poisson(NROW, args.ncol_c2, 0.07, seed=2,
                                   na_rate=1e-6)
    res["c2_nnz"] = x.nnz
    hs = []

    def fresh():
        while hs:
            hs.pop().free()
        hs.append(DeviceSVT(x.nrow, x.nleaf, x.nnz, x.val_type, x.leaf_ptr,
                            x.offs, x.vals))
    ms = timed(lambda: hs[-1].colstats("sum", na_rm=True), args.reps, fresh)
    while hs:
        hs.pop().free()
    record("C2 colSums (wide)", ms, x.nnz * 4.0 + 8.0 * (x.nleaf + 1))
    medians_workloads("C2", x, 4, True)
    res["c2_colMedians_over_colSums_wide"] = (
        res["ops"]["C2 colMedians"]["ms"] / res["ops"]["C2 colSums (wide)"]
        ["ms"])
    del x
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    L.svtgpu_release_cached_memory()

    # --- 3, 4: d = 0.6 -------------------------------------------------
    x = DeviceSVT.generate_poisson(NROW, args.ncol_d6, 0.6, seed=11,
                                   na_rate=1e-6)
    res["d6_nnz"] = x.nnz
    medians_workloads("d0.6", x, 4, True)
    cs = x.colstats("sum", na_rm=True)[0].cpu().numpy()
    sf = cs / cs.mean()
    z = x.ewise("/", sf, margin=2).ewise("log1p")
    del x
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    medians_workloads("d0.6 log1p(x/sf)", z, 8, False)
    del z
    print(json.dumps(res))
    return 0


if __name__ == "__main__":
    sys.exit(main())
