"""Wide and compact kernels of the headline step on the C2 shard (33,538 x
1,000,000 integer counts at density 0.07, nnz = 2.348e9, generated in HBM).

For colSums, colMeans, rowSums and rowVars (na.rm = TRUE) it reports the
kernel time of the op's statistic kernel, from torch.profiler:

  wide      the first call on a fresh handle (int32 offsets and values);
  compact   later calls on a handle that holds the compact copy (uint16
            offsets, int8 values, DESIGN.md section 3);

with the bytes each form reads per call and the GB/s over those bytes (and
the fraction of the 6546 GB/s measured copy bandwidth).  Also the build: the
time of the call that builds the copy, its kernels, and the extra HBM.  The
card's name and power limit are printed with the numbers.  Prints one JSON
line after a table.

    python tools/bench_compact.py [--ncol N] [--reps R]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NROW, DENSITY, SEED, NA_RATE = 33538, 0.07, 2, 1e-6
PEAK_GBS = 6546.0
OPS = ("colSums", "colMeans", "rowSums", "rowVars")
# the statistic kernels of each op (finalize kernels and memsets excluded)
HOT = ("colstats_direct", "colstats_sum_i8", "row_hist<")


def device_card():
    try:
        out = subprocess.run(
            ["nvidia-smi", "--query-gpu=name,power.limit",
             "--format=csv,noheader"], capture_output=True, text=True,
            timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:          # the query is informative only
        return "unknown (%s)" % e


def run_op(d, op):
    if op == "colSums":
        return d.colstats("sum", na_rm=True)[0]
    if op == "colMeans":
        return d.colstats("mean", na_rm=True)[0]
    if op == "rowSums":
        return d.rowstats("sum", na_rm=True)[0]
    return d.rowmoments(na_rm=True)[1]


def kernel_ms(calls):
    """{kernel name: total device ms} of the kernels the calls launch"""
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for fn in calls:
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        out[ev.name] = out.get(ev.name, 0.0) + ev.device_time_total / 1e3
    return out


def hot_ms(k):
    return sum(v for n, v in k.items() if any(h in n for h in HOT))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--ncol", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()

    import torch
    from sparsearray_b200 import _native as N
    from sparsearray_b200.device import DeviceSVT
    if N.device_count() < 1:
        raise SystemExit("bench_compact.py: no CUDA device")

    x = DeviceSVT.generate_poisson(NROW, args.ncol, DENSITY, seed=SEED,
                                   na_rate=NA_RATE)
    nnz, nleaf = x.nnz, x.nleaf

    def fresh():
        return DeviceSVT(NROW, nleaf, nnz, "integer", x.leaf_ptr, x.offs,
                         x.vals)

    def compact_bytes(d):
        b = ctypes.c_int64(0)
        N.check(N.lib().svtgpu_matrix_compact_bytes(d._h, ctypes.byref(b)))
        return b.value

    def read_bytes(op, entry_bytes):
        col = op.startswith("col")
        return nnz * entry_bytes + (8 * (nleaf + 1) if col else 0)

    # every kernel and cache once (the max |x| pass, the tile table)
    for op in OPS:
        run_op(x, op)
    x.free()

    res = {}
    # wide: the first call of a fresh handle, which builds nothing
    for op in OPS:
        hs = [fresh() for _ in range(args.reps)]
        # (a fresh handle's row call also runs the max |x| pass and builds
        # the tile table: those kernels are not counted)
        k = kernel_ms([lambda h=h: run_op(h, op) for h in hs])
        assert all(compact_bytes(h) == 0 for h in hs)
        for h in hs:
            h.free()
        res[op] = {"wide_ms": hot_ms(k) / args.reps,
                   "wide_bytes": read_bytes(op, 4 if op.startswith("col")
                                            else 8)}

    # the build: second eligible call on a fresh handle
    d = fresh()
    run_op(d, "colSums")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    kb = kernel_ms([lambda: run_op(d, "colSums")])
    build_call_ms = (time.perf_counter() - t0) * 1e3
    extra = compact_bytes(d)
    assert extra > 0, "the compact copy was not built"
    build = {"call_ms_host_clock": build_call_ms,
             "kernels_ms": {n: v for n, v in kb.items()
                            if "memset" not in n.lower()},
             "extra_hbm_bytes": extra}

    for op in OPS:
        run_op(d, op)
        k = kernel_ms([lambda: run_op(d, op)] * args.reps)
        res[op]["compact_ms"] = hot_ms(k) / args.reps
        res[op]["compact_bytes"] = read_bytes(op, 1 if op.startswith("col")
                                              else 3)
    d.free()

    card = device_card()
    print("card: %s   nnz = %d   reps = %d" % (card, nnz, args.reps))
    print("%-9s %9s %9s %8s %11s %11s %6s %6s" % (
        "op", "wide ms", "cmp ms", "speedup", "wide GB/s", "cmp GB/s",
        "wfrac", "cfrac"))
    for op in OPS:
        r = res[op]
        r["wide_GBps"] = r["wide_bytes"] / (r["wide_ms"] * 1e-3) / 1e9
        r["compact_GBps"] = r["compact_bytes"] / (r["compact_ms"] * 1e-3) / 1e9
        r["speedup"] = r["wide_ms"] / r["compact_ms"]
        print("%-9s %9.3f %9.3f %8.2f %11.0f %11.0f %6.2f %6.2f" % (
            op, r["wide_ms"], r["compact_ms"], r["speedup"], r["wide_GBps"],
            r["compact_GBps"], r["wide_GBps"] / PEAK_GBS,
            r["compact_GBps"] / PEAK_GBS))
    print("build: second call %.1f ms (host clock), kernels %s, extra HBM "
          "%.2f GB" % (build_call_ms, json.dumps(
              {n: round(v, 3) for n, v in build["kernels_ms"].items()}),
              extra / 1e9))
    print(json.dumps({"card": card, "nnz": nnz, "reps": args.reps,
                      "peak_GBps": PEAK_GBS, "ops": res, "build": build}))


if __name__ == "__main__":
    main()
