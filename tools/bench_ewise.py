"""Element-wise operations on the C2 shape (33,538 x 1,000,000 integer counts
at density 0.07, nnz = 2.348e9, generated in HBM): CUDA-event times of

  sweep(x, 2, sf, "/")     integer -> double    (sf = colSums / mean)
  log1p(y)                 double  -> double
  x * 2L                   integer -> integer
  floor(x / 3)             the compaction path (timed: floor of x / 3)
  rowMoments(log1p(sweep(x, 2, sf, "/")))      the whole pipeline

each with its algorithmic bytes (from nnz: offsets + values read and
written, 16 B per leaf) and the fraction of the 6546 GB/s measured copy
bandwidth; the host alternative on the first 100,000 columns (numpy
transform of the CSC, then from_csc); a parity check against the oracle on
the first and last 1,000 columns.  Prints one JSON line.

    python tools/bench_ewise.py [--ncol N] [--reps R]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))   # the ewise oracle

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncol", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-cols", type=int, default=100_000)
    args = ap.parse_args()
    import torch
    import sparsearray_b200 as sa
    import ewise_oracle
    from oracle import port
    from sparsearray_b200 import synth
    from sparsearray_b200.device import DeviceSVT

    ncol = args.ncol
    x = DeviceSVT.generate_poisson(NROW, ncol, DENSITY, seed=SEED,
                                   na_rate=NA_RATE)
    nnz = x.nnz
    cs, _ = x.colstats("sum", na_rm=True)
    cs = cs.cpu().numpy()
    sf = cs / cs.mean()
    leaf_bytes = 16.0 * ncol

    def gb(read_v, write_v):
        return (nnz * (4 + read_v + 4 + write_v) + leaf_bytes) / 1e9

    res = {"device": device_card(), "shape": [NROW, ncol], "nnz": nnz,
           "peak_copy_GBs": PEAK_GBS, "ops": {}}
    keep = {}

    def op_sweep():
        keep["y"] = x.ewise("/", sf, margin=2)

    def op_log1p():
        keep["z"] = keep["y"].ewise("log1p")

    def op_mul2():
        keep["m"] = x.ewise("*", np.array([2], np.int32))

    def op_floor():
        keep["f"] = keep["d3"].ewise("floor")

    cases = [("sweep_div_int_to_double", op_sweep, gb(4, 8)),
             ("log1p_double", op_log1p, gb(8, 8)),
             ("mul_2L_int", op_mul2, gb(4, 4))]
    for name, fn, g in cases:
        med, lo, hi = timed(fn, args.reps)
        res["ops"][name] = {"ms": med, "ms_min": lo, "ms_max": hi,
                            "alg_GB": g, "GBs": g / med * 1e3,
                            "frac_peak": g / med * 1e3 / PEAK_GBS}
    keep.pop("m", None)
    keep["d3"] = x.ewise("/", np.array([3.0]))
    med, lo, hi = timed(op_floor, args.reps)
    f = keep["f"]
    g = (nnz * 24 + f.nnz * 12 + leaf_bytes * 3) / 1e9   # map + count + copy
    res["ops"]["floor_div3_compaction"] = {
        "ms": med, "ms_min": lo, "ms_max": hi, "alg_GB": g,
        "GBs": g / med * 1e3, "frac_peak": g / med * 1e3 / PEAK_GBS,
        "nnz_in": nnz, "nnz_out": f.nnz}
    del keep["d3"], keep["f"]

    def pipeline():
        y = x.ewise("/", sf, margin=2)
        z = y.ewise("log1p")
        del y
        keep["mv"] = z.rowmoments()
        del z

    med, lo, hi = timed(pipeline, max(2, args.reps // 2))
    res["ops"]["pipeline_rowMoments_log1p_sweep"] = {"ms": med, "ms_min": lo,
                                                     "ms_max": hi}

    # parity: column statistics of the device results on the first and last
    # 1,000 columns against the oracle's transformed CSC
    y, z = keep["y"], keep["z"]
    ok = True
    stats = {}
    for nm, h in (("y", y), ("z", z)):
        stats[nm] = {op: h.colstats(op)[0].cpu().numpy()
                     for op in ("max", "min", "countNAs", "sum")}
    for l0 in (0, ncol - 1000):
        p, o, v = synth.poisson_csc(NROW, 1000, DENSITY, seed=SEED,
                                    na_rate=NA_RATE, leaf0=l0)
        ty = ewise_oracle.ewise(NROW, 1000, p, o, v, "integer", "/",
                        sf[l0:l0 + 1000], "double", 2)
        tz = ewise_oracle.ewise(NROW, 1000, *ty[:3], "double", "log1p")
        for nm, t in (("y", ty), ("z", tz)):
            for op in ("max", "min", "countNAs", "sum"):
                exp = port.colstats(NROW, 1000, *t[:3], "double", op)[0]
                got = stats[nm][op][l0:l0 + 1000]
                m = ~np.isnan(exp)
                same_nan = np.array_equal(np.isnan(got), np.isnan(exp))
                if nm == "y" and op != "sum":
                    good = same_nan and np.array_equal(got[m], exp[m])
                else:
                    good = same_nan and np.allclose(got[m], exp[m],
                                                    rtol=1e-12, atol=0)
                ok = ok and bool(good)
    res["parity_first_last_1000_cols"] = ok
    del keep["y"], keep["z"]

    # host alternative: numpy transform of the CSC, then from_csc
    hc = min(args.host_cols, ncol)
    p, o, v = synth.poisson_csc(NROW, hc, DENSITY, seed=SEED,
                                na_rate=NA_RATE)
    t0 = time.perf_counter()
    cols = np.repeat(np.arange(hc), np.diff(p))
    na = v == sa.NA_INTEGER
    with np.errstate(invalid="ignore"):
        w = np.log1p(v / sf[cols])
    w[na] = sa.NA_REAL
    t1 = time.perf_counter()
    r = sa.from_csc((NROW, hc), p, w, o)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    r.release()
    res["host_alternative"] = {
        "cols": hc, "transform_ms": (t1 - t0) * 1e3,
        "from_csc_ms": (t2 - t1) * 1e3,
        "device_equivalent_ms": (res["ops"]["sweep_div_int_to_double"]["ms"]
                                 + res["ops"]["log1p_double"]["ms"])
        * hc / ncol}
    print(json.dumps(res))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
