#!/usr/bin/env python
"""Benchmark of the SVT hot path: every configuration BASELINE.json names.

Headline (`value`, BASELINE configs[1] = "C2"): per GPU a 33,538 x 1,000,000
integer count matrix at density 0.07 (poissonSparseArray distribution, NAs
injected at 1e-6), resident in HBM as a device CSC.  One *step* = colSums,
colMeans, rowSums and rowVars of it, all with na.rm=TRUE; `value` = nonzeros
processed per second over the whole job (4 passes x nnz per step).  Weak
scaling: every rank owns its own 1,000,000 columns of a 33,538 x
(N x 1,000,000) matrix; row-shaped results are allreduced (NCCL).  Inputs
(18.8 GB per rank) are far larger than L2, so no L2 flush between iterations.

The other configurations hang off keys the driver keeps:

  roofline.per_op[...]        device-timed kernels of every op / config: ms,
                              nnz/s, algorithmic GB/s, fraction of the
                              measured HBM peak (C2 incl. the atomic-free row
                              kernels, C3 products, C1, C5, C2 values as double)
  roofline.strong_scaling_c4  configs[3] as written: ONE 33,538 x 4,000,000
                              matrix column-sharded over the N ranks
  e2e.per_config[...]         the same ops through the `.Call` entry points
                              from HOST buffers (flatten + H2D + kernels + D2H)
  cpu_baseline.per_config[..] the reference's own C (oracle/_ref) on all host
                              cores, N = 1 only, bounded samples
  config.parity_checked       in-bench parity of the timed kernels against the
                              reference's outputs (the run FAILS on mismatch)

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N
    python bench.py --impl reference      # the reference's CPU code, host cores
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NROW = 33538
NCOL_PER_GPU = 1_000_000
DENSITY = 0.07
NA_RATE = 1e-6
SEED = 2
K_DENSE = 50
C4_TOTAL_COLS = 4_000_000
C1_DIM, C1_DENSITY = (20000, 5000), 0.05
C5_NROW, C5_NCOL, C5_DENSITY = 100_000, 2_000_000, 0.01
MIN_WARMUP = 32
# --dump-outputs stays below 64 MB in all, .npy headers included
DUMP_BYTES = 63 * 10**6
METRIC = "nnz/s for SVT colSums+colMeans+rowSums+rowVars (na.rm=TRUE), " \
         "33538x1e6 int counts d=0.07 per GPU"
OPS = ["colSums", "colMeans", "rowSums", "rowVars"]


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / event reasons of one GPU during the timed region.

    nvidia-smi needs ~0.1 s to start, more than a short timed region lasts, so
    it is started before the warm-up steps and every sample carries its time
    stamp: stop(t0, t1) keeps the samples taken inside the timed region and,
    when the region was too short to hold two, the ones taken under the same
    load during the warm-up just before it (noted in the result)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,"
         "clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
             "sw_power_cap"]

    def __init__(self, index):
        self.p = None
        self.path = "/tmp/svt_clocks_%d_%d.csv" % (os.getpid(), index)
        try:
            self.f = open(self.path, "w")
            self.p = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    @staticmethod
    def _epoch(stamp):
        import datetime
        try:
            return datetime.datetime.strptime(
                stamp.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self, t0=None, t1=None):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [],
               "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.close()
        rows = []
        try:
            for line in open(self.path):
                parts = [x.strip() for x in line.split(",")]
                if len(parts) < 8:
                    continue
                try:
                    rows.append((self._epoch(parts[0]), float(parts[1]),
                                 float(parts[2]), parts[4:8]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except Exception:
            pass
        inside = rows
        if t0 is not None and t1 is not None:
            inside = [r for r in rows if r[0] is not None and
                      t0 <= r[0] <= t1]
            if len(inside) < 2:
                # short region: the warm-up steps right before it ran the
                # same kernels back to back
                inside = [r for r in rows if r[0] is not None and
                          t0 - 3.0 <= r[0] <= t1 + 0.05]
                out["note"] = ("timed region shorter than the sampling "
                               "interval: samples from the warm-up steps "
                               "just before it included")
        reasons = set()
        for r in inside:
            for name, val in zip(self.NAMES, r[3]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if inside:
            out["sm_mhz"] = statistics.median(r[1] for r in inside)
            out["sm_max_mhz"] = max(r[2] for r in inside)
            out["samples"] = len(inside)
        out["reasons"] = sorted(reasons)
        return out


def algorithmic_bytes(op, nnz, nleaf, nrow, vsz=4):
    """SURVEY.md section 8(d): bytes one launch must move.  vsz = bytes per
    stored value (4 int, 8 double, 0 lacunar)."""
    if op.startswith("col"):
        return nnz * vsz + (nleaf + 1) * 8 + nleaf * 8
    slots = 4 if op == "rowVars" else 3
    return nnz * (4 + vsz) + (nleaf + 1) * 8 + nrow * 8 * (slots + 1)


def product_bytes(nnz, nleaf, nrow, K):
    """crossprod / %*%: the SVT once (offsets + double values), the dense
    operand once, the result once"""
    return nnz * 12 + (nleaf + 1) * 8 + (nrow + nleaf) * K * 8


def entry(ms, nnz, nbytes, peak, **extra):
    e = {"ms": round(ms, 4), "nnz_per_s": nnz / (ms * 1e-3),
         "GBps": nbytes / (ms * 1e-3) / 1e9,
         "frac": nbytes / (ms * 1e-3) / 1e9 / peak}
    e.update(extra)
    return e


def host_copy_bandwidth(nbytes, nthreads):
    """GB/s (bytes read + bytes written) of a plain multi-threaded copy
    between two pageable host arrays: the ceiling for the flatten, which
    gathers leaf payloads into the pinned staging slots"""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    n = max(1, nbytes // 8)
    src = np.ones(n, dtype=np.float64)
    dst = np.empty(n, dtype=np.float64)
    cuts = [(n * i) // nthreads for i in range(nthreads + 1)]

    def part(i):
        np.copyto(dst[cuts[i]:cuts[i + 1]], src[cuts[i]:cuts[i + 1]])

    best = 1e30
    with ThreadPoolExecutor(nthreads) as ex:
        for _ in range(3):
            t0 = time.perf_counter()
            list(ex.map(part, range(nthreads)))
            best = min(best, time.perf_counter() - t0)
    return 2 * n * 8 / best / 1e9


def best_wall(fn, n=3, warm=1):
    for _ in range(warm):
        fn()
    best = 1e30
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return best


# ---------------------------------------------------------------------------
# the reference's own CPU implementation (oracle/_ref, built from the
# reference's sources) on the host cores.  These legs and the in-bench parity
# check are the only places this file touches oracle/.

def host_sample(ncols, seed=SEED):
    """Columns [0, ncols) of the C2 matrix as a host SVT_SparseMatrix.
    Generated on the GPU when there is one (same formula), else on the host."""
    from sparsearray_b200 import synth, _native
    from sparsearray_b200.svt import SVT_SparseArray
    if _native.device_count() > 0:
        import torch
        from sparsearray_b200.device import DeviceSVT
        d = DeviceSVT.generate_poisson(NROW, ncols, DENSITY, seed=seed,
                                       na_rate=NA_RATE)
        ptr = d.leaf_ptr.cpu().numpy()
        offs = d.offs[:d.nnz].cpu().numpy()
        vals = d.vals[:d.nnz].cpu().numpy()
        del d
        torch.cuda.empty_cache()
        return SVT_SparseArray((NROW, ncols), "integer", ptr, offs, vals)
    return synth.poisson_svt(NROW, ncols, DENSITY, seed=seed,
                             na_rate=NA_RATE)


def host_lacunar_sample(ncols, seed=5):
    from sparsearray_b200 import synth, _native
    from sparsearray_b200.svt import SVT_SparseArray
    if _native.device_count() > 0:
        import torch
        from sparsearray_b200.device import DeviceSVT
        d = DeviceSVT.generate_poisson(C5_NROW, ncols, C5_DENSITY, seed=seed,
                                       lacunar=True)
        ptr = d.leaf_ptr.cpu().numpy()
        offs = d.offs[:d.nnz].cpu().numpy()
        del d
        torch.cuda.empty_cache()
        return SVT_SparseArray((C5_NROW, ncols), "integer", ptr, offs, None)
    return synth.poisson_svt(C5_NROW, ncols, C5_DENSITY, seed=seed,
                             lacunar=True)


def dense_operands(ncols, seed=7):
    """Y (NROW x K) and D (ncols x K), N(0, 1), column-major as in R"""
    import numpy as np
    rng = np.random.Generator(np.random.PCG64(seed))
    Y = np.asfortranarray(rng.standard_normal((NROW, K_DENSE)))
    D = np.asfortranarray(rng.standard_normal((ncols, K_DENSE)))
    return Y, D


def reference_step(x):
    """The four ops exactly as the reference's R methods run them: colSums,
    colMeans: one C_colStats_SVT call each (OpenMP over columns); rowSums: one
    serial C_rowStats_SVT call; rowVars: three (countNAs, sum,
    centered_X2_sum) + R arithmetic.  Returns the four results."""
    from oracle import refcall
    return (refcall.colStats(x, "sum", na_rm=True).value,
            refcall.colStats(x, "mean", na_rm=True).value,
            refcall.rowStats(x, "sum", na_rm=True).value,
            refcall.rowVars(x, na_rm=True))


def sparse_crossprod_inputs():
    """The shapes of the reference's own benchmark script
    (inst/scripts/benchmark_crossprod.R:143-166): svt1 25000 x 400 at density
    0.07 and svt2 25000 x 650 at density 0.20, double."""
    import numpy as np
    from sparsearray_b200.svt import SVT_SparseArray
    rng = np.random.Generator(np.random.PCG64(11))

    def make(nrow, ncol, density):
        cnt = rng.binomial(nrow, density, size=ncol)
        ptr = np.zeros(ncol + 1, dtype=np.int64)
        np.cumsum(cnt, out=ptr[1:])
        offs = np.concatenate([np.sort(rng.choice(nrow, size=c,
                                                  replace=False))
                               for c in cnt]).astype(np.int32)
        vals = np.round(rng.standard_normal(offs.size), 2)
        vals[vals == 0] = 0.5
        return SVT_SparseArray((nrow, ncol), "double", ptr, offs, vals)
    return make(25000, 400, 0.07), make(25000, 650, 0.20)


def time_sparse_crossprod(fn1, fn2):
    """seconds (best of 3) of crossprod(svt1), crossprod(svt1, svt2) and
    crossprod(svt2, svt1) with the given unary / binary implementations"""
    s1, s2 = sparse_crossprod_inputs()
    s1.r_SVT, s2.r_SVT
    out = {}
    for name, f in (("crossprod(svt1)", lambda: fn1(s1)),
                    ("crossprod(svt1, svt2)", lambda: fn2(s1, s2)),
                    ("crossprod(svt2, svt1)", lambda: fn2(s2, s1))):
        out[name] = round(best_wall(f), 4)
    s1.release()
    s2.release()
    return out


def cpu_c2(ncols, steps, warmup=1):
    """(cpu_baseline dict, outputs of the last step, the host sample)"""
    from oracle import refcall
    if not refcall.available():
        raise RuntimeError("oracle/_ref/libsvtref.so is missing")
    cores = refcall.num_procs()
    refcall.set_threads(cores)     # set_SparseArray_nthread(<all cores>)
    x = host_sample(ncols)
    x.r_SVT   # build the leaf list outside the timed region
    for _ in range(warmup):
        reference_step(x)
    times = []
    outs = None
    for _ in range(steps):
        t0 = time.perf_counter()
        outs = reference_step(x)
        times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    nnz = x.nnz
    base = {"value": len(OPS) * nnz / t, "unit": "nnz/s", "cores": cores,
            "kind": "reference",
            "sample": "first %d of 1e6 columns (nnz=%d), %d steps of the "
                      "same 4 ops through the reference's .Call entry points "
                      "(oracle/_ref), OpenMP threads = all %d host cores; "
                      "rowStats is serial in the reference"
                      % (ncols, nnz, steps, cores),
            "ms_per_step": t * 1e3}
    return base, outs, x


def cpu_other_configs(x_c2, prod_cols, c5_cols, skip=()):
    """cpu_baseline.per_config: the reference on bounded samples of the other
    configurations.  x_c2 = the host C2 sample (its first prod_cols columns,
    as double, are the C3 sample).  Returns (per_config, outputs) --
    outputs are compared with the GPU's on the same inputs by the caller."""
    import numpy as np
    from oracle import refcall
    from sparsearray_b200 import synth
    from sparsearray_b200.svt import SVT_SparseArray
    cores = refcall.num_procs()
    refcall.set_threads(cores)
    per, outs = {}, {}

    if "C3" not in skip:
        # ---- C3: crossprod(svt, Y) and svt %*% D on the first prod_cols
        # columns (double), all cores; the reference makes K passes over the
        # SVT (src/SparseMatrix_mult.c:385-431, OpenMP loop :143-152) and
        # `%*%` transposes first (R/SparseMatrix-mult.R:196-198)
        e1 = int(x_c2.ptr[prod_cols])
        xs = SVT_SparseArray((NROW, prod_cols), "integer",
                             x_c2.ptr[:prod_cols + 1], x_c2.offs[:e1],
                             x_c2.vals[:e1]).with_type("double")
        xs.r_SVT
        Y, D = dense_operands(prod_cols)
        t = best_wall(lambda: refcall.crossprod2_SVT_mat(xs, Y), n=2, warm=1)
        outs["crossprod"] = refcall.crossprod2_SVT_mat(xs, Y).value
        per["C3 crossprod(svt, Y[33538x50])"] = {
            "value": xs.nnz / t, "unit": "nnz/s", "seconds": round(t, 4),
            "sample": "first %d columns as double (nnz=%d), "
                      "C_crossprod2_SVT_mat, %d cores" % (prod_cols, xs.nnz,
                                                          cores)}
        t = best_wall(lambda: refcall.matmul_SVT_mat(xs, D), n=2, warm=1)
        outs["matmul"] = refcall.matmul_SVT_mat(xs, D).value
        tt = best_wall(lambda: refcall.transpose_2D_SVT(xs).release(), n=1,
                       warm=0)
        per["C3 svt %*% D[ncol x 50]"] = {
            "value": xs.nnz / t, "unit": "nnz/s", "seconds": round(t, 4),
            "transpose_seconds": round(tt, 4),
            "sample": "first %d columns as double (nnz=%d), D = its %d rows: "
                      "C_transpose_2D_SVT (serial) + C_crossprod2_SVT_mat, "
                      "%d cores" % (prod_cols, xs.nnz, prod_cols, cores)}
        outs["c3_sample"] = xs

    if "C1" not in skip:
        # ---- C1: the reference's own CPU-runnable case, full size
        x1 = synth.random_svt(C1_DIM[0], C1_DIM[1], C1_DENSITY, seed=1)
        x1.r_SVT
        c1 = {}
        for name, f in (
                ("colSums", lambda: refcall.colStats(x1, "sum")),
                ("colVars", lambda: refcall.colStats(x1, "var1")),
                ("rowSums", lambda: refcall.rowStats(x1, "sum")),
                ("rowVars", lambda: refcall.rowVars(x1))):
            c1[name] = {"ms": round(best_wall(f, n=5) * 1e3, 4)}
            r = f()
            outs["C1 " + name] = r.value if hasattr(r, "value") else r
        per["C1 20000x5000 double d=0.05 (nnz=%d)" % x1.nnz] = {
            "ops": c1, "sample": "full size, best of 5, %d cores" % cores}
        outs["c1_matrix"] = x1

    if "C5" not in skip:
        # ---- C5: lacunar, first c5_cols of the 2e6 columns
        x5 = host_lacunar_sample(c5_cols)
        x5.r_SVT
        c5 = {}
        for name, f in (
                ("colSums", lambda: refcall.colStats(x5, "sum")),
                ("rowSums", lambda: refcall.rowStats(x5, "sum")),
                ("rowVars", lambda: refcall.rowVars(x5))):
            t = best_wall(f, n=2, warm=1)
            c5[name] = {"ms": round(t * 1e3, 3), "nnz_per_s": x5.nnz / t}
            r = f()
            outs["C5 " + name] = r.value if hasattr(r, "value") else r
        per["C5 lacunar 100000 x 2e6 d=0.01"] = {
            "ops": c5, "sample": "first %d columns (nnz=%d), %d cores"
                                 % (c5_cols, x5.nnz, cores)}
        outs["c5_sample"] = x5
    return per, outs


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncols = args.cpu_cols
    steps = max(1, min(args.steps, 5))
    base, _, x = cpu_c2(ncols, steps, warmup=min(args.warmup, 1))
    try:
        per, outs = cpu_other_configs(x, args.cpu_prod_cols, args.cpu_c5_cols)
        for k in ("c3_sample", "c1_matrix", "c5_sample"):
            if k in outs:
                outs[k].release()
    except Exception as e:
        per = {"error": str(e)}
    try:   # the reference's own (sparse x sparse) benchmark shapes, seconds
        from oracle import refcall
        per["sparse_crossprod_s (benchmark_crossprod.R shapes)"] = \
            time_sparse_crossprod(refcall.crossprod1_SVT,
                                  refcall.crossprod2_SVT_SVT)
    except Exception as e:
        per["sparse_crossprod_s"] = {"error": str(e)}
    x.release()
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"],
        "unit": "nnz/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": min(args.warmup, 1), "ms_per_step": base["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32->f64", "data": "synthetic",
        "config": {"workload": "configs[1]: 33538x1e6 int counts d=0.07, "
                               "colSums/colMeans/rowSums/rowVars na.rm=TRUE",
                   "sample_cols": ncols},
        "cpu_baseline": {"value": base["value"], "unit": "nnz/s",
                         "cores": base["cores"], "kind": "reference",
                         "sample": base["sample"], "per_config": per},
        "e2e": {"value": base["value"], "unit": "nnz/s",
                "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------
# outputs of the timed step, for comparing two builds on the same inputs

def dump_outputs(path, last, rank, world):
    """Write the results of the last timed step as <path>/<op>.npy (float64).
    Row results are allreduced, so rank 0 writes them; every rank writes its
    own columns (<op>_rank<r>.npy when there are several).  Beyond
    DUMP_BYTES in all, the column results are cut to the same fixed, seeded
    sample of columns on every run."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    out = {op: np.asarray(t.cpu().numpy(), dtype=np.float64)
           for op, t in last.items()}
    col_ops = [op for op in OPS if op.startswith("col")]
    row_bytes = sum(out[op].nbytes for op in OPS if op.startswith("row"))
    ncol = out[col_ops[0]].size
    keep = (DUMP_BYTES - row_bytes) // (8 * len(col_ops) * world)
    pick = None
    if ncol > keep:
        pick = np.sort(np.random.Generator(np.random.PCG64(0)).choice(
            ncol, size=keep, replace=False))
    for op in OPS:
        if op in col_ops:
            a = out[op] if pick is None else out[op][pick]
            name = op if world == 1 else "%s_rank%d" % (op, rank)
        elif rank == 0:
            a, name = out[op], op
        else:
            continue
        np.save(os.path.join(path, name + ".npy"), a)


# ---------------------------------------------------------------------------
# in-bench parity

class ParityError(RuntimeError):
    pass


def _same(name, got, exp, rtol=0.0, cond=None):
    """NA/NaN pattern identical; values bit-equal (rtol 0) or within rtol of
    max(|expected|, cond).  cond = sum of |terms| for sums of signed terms
    (their condition: a differently ordered sum of cancelling terms is only
    defined to n * eps * sum|x|)"""
    import numpy as np
    got = np.asarray(got, dtype=np.float64).reshape(-1)
    exp = np.asarray(exp, dtype=np.float64).reshape(-1)
    if got.shape != exp.shape:
        raise ParityError("%s: shape %s vs %s" % (name, got.shape, exp.shape))
    if not np.array_equal(np.isnan(got), np.isnan(exp)):
        raise ParityError("%s: NA/NaN pattern differs" % name)
    m = ~np.isnan(exp)
    if rtol == 0.0:
        if not np.array_equal(got[m], exp[m]):
            bad = int(np.flatnonzero(got[m] != exp[m])[0])
            raise ParityError("%s: not bit-exact (first at %d: %r vs %r)"
                              % (name, bad, got[m][bad], exp[m][bad]))
        return 0.0
    with np.errstate(all="ignore"):
        fin = m & np.isfinite(exp)
        if not np.array_equal(got[m & ~fin], exp[m & ~fin]):
            raise ParityError("%s: infinities differ" % name)
        scale = np.maximum(np.abs(exp[fin]), 1e-300)
        if cond is not None:
            scale = np.maximum(scale, np.asarray(cond,
                                                 dtype=np.float64).reshape(-1)[fin])
        err = np.abs(got[fin] - exp[fin]) / scale
    worst = float(err.max()) if err.size else 0.0
    if worst > rtol:
        raise ParityError("%s: relative error %.3g > %.1g" % (name, worst,
                                                              rtol))
    return worst


# ---------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--cols", type=int, default=NCOL_PER_GPU,
                    help="columns per GPU (default: the full workload)")
    ap.add_argument("--cpu-cols", type=int, default=100_000,
                    help="columns of the bounded CPU-baseline sample (C2)")
    ap.add_argument("--cpu-prod-cols", type=int, default=20_000,
                    help="columns of the CPU sample of the C3 products")
    ap.add_argument("--cpu-c5-cols", type=int, default=100_000)
    ap.add_argument("--e2e-cols", type=int, default=None,
                    help="columns per GPU of the end-to-end leg "
                         "(default: all)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--c5-cols", type=int, default=C5_NCOL)
    ap.add_argument("--c4-cols", type=int, default=C4_TOTAL_COLS)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-products", action="store_true")
    ap.add_argument("--no-configs", action="store_true",
                    help="skip the C1 / C5 / C4 legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step "
                         "(colSums, colMeans, rowSums, rowVars) as "
                         "DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    import sparsearray_b200 as sa
    from sparsearray_b200 import _native as N
    from sparsearray_b200 import sharded, rcall
    from sparsearray_b200.device import DeviceSVT
    from sparsearray_b200.svt import SVT_SparseArray

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if N.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device (there is no CPU path)")
    torch.cuda.set_device(local)
    N.check(N.lib().svtgpu_set_device(local))
    group_cpu = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        group_cpu = dist.new_group(backend="gloo")
    dev = torch.device("cuda", local)
    grp = dist.group.WORLD if world > 1 else None
    peak, peak_kind = hbm_peak()
    warmup = max(args.warmup, MIN_WARMUP)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def dev_ms(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        barrier()
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        barrier()
        return a.elapsed_time(b) / reps

    def maxr(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def sumr(v):
        t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.item()

    def env_set(**kv):
        old = {k: os.environ.get(k) for k in kv}
        for k, v in kv.items():
            os.environ[k] = v
        return old

    def env_restore(old):
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v

    # =====================================================================
    # C2: the headline step
    ncol = args.cols
    shard = DeviceSVT.generate_poisson(
        NROW, ncol, DENSITY, seed=SEED, na_rate=NA_RATE, leaf0=rank * ncol,
        nleaf_total=world * ncol)
    nnz = shard.nnz

    # preallocated outputs / states (steady-state serving: no allocation in
    # the timed region)
    col_out = torch.empty(ncol, dtype=torch.float64, device=dev)
    col_warn = torch.zeros(4, dtype=torch.int32, device=dev)
    st3 = torch.empty(6 * NROW, dtype=torch.float64, device=dev)
    st4 = torch.empty(6 * NROW, dtype=torch.float64, device=dev)

    def run_op(op, s=None, g=grp):
        s = shard if s is None else s
        if op == "colSums":
            return s.colstats("sum", na_rm=True, out=col_out[:s.nleaf],
                              warn=col_warn)[0]
        if op == "colMeans":
            return s.colstats("mean", na_rm=True, out=col_out[:s.nleaf],
                              warn=col_warn)[0]
        if op == "rowSums":
            return s.rowstats("sum", na_rm=True, group=g, state=st3)[0]
        return s.rowmoments(na_rm=True, group=g, state=st4)[1]

    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(len(OPS) + 1)]
          for _ in range(args.steps)]
    sampler = ClockSampler(local) if rank == 0 else None
    # at least MIN_WARMUP steps (~0.3 s) of the same load before the timed
    # region: nvidia-smi's start-up, and cover for timed regions shorter than
    # its sampling interval (the same count on every rank: the row
    # operations are collectives)
    for _ in range(warmup):
        for op in OPS:
            run_op(op)
    # --dump-outputs: the last step's results are copied aside in stream
    # order as they come (colSums and colMeans share col_out)
    last = None
    if args.dump_outputs:
        last = {op: torch.empty(ncol if op.startswith("col") else NROW,
                                dtype=torch.float64, device=dev)
                for op in OPS}
    barrier()
    launches0 = N.launch_count()
    t_begin = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    wall0 = time.time()
    t_begin.record()
    for s in range(args.steps):
        ev[s][0].record()
        for i, op in enumerate(OPS):
            if last is not None and s == args.steps - 1:
                last[op].copy_(run_op(op))
            else:
                run_op(op)
            ev[s][i + 1].record()
    t_end.record()
    barrier()
    wall1 = time.time()
    launches = N.launch_count() - launches0
    clocks = sampler.stop(wall0, wall1) if sampler else None
    if last is not None:
        dump_outputs(args.dump_outputs, last, rank, world)
    per_op_ms = [sum(ev[s][i].elapsed_time(ev[s][i + 1])
                     for s in range(args.steps)) / args.steps
                 for i in range(len(OPS))]
    total_ms = maxr(t_begin.elapsed_time(t_end))
    nnz_total = sumr(nnz)
    ms_per_step = total_ms / args.steps
    value = len(OPS) * nnz_total / (ms_per_step * 1e-3)

    per_op = {}
    for op, ms in zip(OPS, per_op_ms):
        per_op["C2 " + op] = entry(ms, nnz, algorithmic_bytes(op, nnz, ncol,
                                                              NROW), peak)
    dom = max(OPS, key=lambda o: per_op["C2 " + o]["ms"])
    roofline = {
        "bound": "hbm", "kernel": {
            "colSums": "colstats_direct<SUM,int>",
            "colMeans": "colstats_direct<SUM,int>",
            "rowSums": "row_hist<SUM32> (shared-memory histogram, cyclic "
                       "tiles, unpredicated double-buffered batches)",
            "rowVars": "row_hist<MOMENTS> (packed sum | sum of squares, "
                       "cyclic tiles) + row_moments_finalize"}[dom],
        "op": dom, "achieved": per_op["C2 " + dom]["GBps"], "peak": peak,
        "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)"
        if peak_kind == "measured" else "fallback",
        "unit": "GB/s", "frac": per_op["C2 " + dom]["frac"],
        "traffic": None, "traffic_source": None,
        "algorithmic_bytes_per_launch": algorithmic_bytes(dom, nnz, ncol,
                                                          NROW),
        "peak_note": "peak = measured COPY bandwidth (read + written bytes); "
                     "a read-only int4 stream reaches ~6.99 TB/s on these "
                     "boxes (tools/microbench/clock_after_stream.cu), so "
                     "read-only kernels can show frac slightly above 1"}
    # DRAM bytes per launch of the dominant kernel from the committed ncu
    # capture (scaled by nonzeros when the capture was of a smaller shard)
    traffic = {}
    try:
        for fn_ in ("r1_traffic.json", "r2_traffic.json"):
            p_ = os.path.join(ROOT, "profiles", fn_)
            if os.path.exists(p_):
                with open(p_) as f:
                    traffic.update(json.load(f))
        tr = traffic.get(dom)
        if tr:
            roofline["traffic"] = tr["bytes"] * (nnz / tr["nnz"])
            roofline["traffic_source"] = tr["capture"] + (
                "" if abs(nnz / tr["nnz"] - 1) < 0.01 else
                "; scaled x%.2f by nonzeros" % (nnz / tr["nnz"]))
    except Exception:
        pass

    # ---- the other reductions of the path, same shard (not in `value`) ---
    def extra(name, fn, op_key, reps=5):
        try:
            ms = dev_ms(fn, reps=reps)
            per_op[name] = entry(ms, nnz, algorithmic_bytes(op_key, nnz, ncol,
                                                            NROW), peak)
        except Exception as e:     # never lose the bench line over an extra
            per_op[name] = {"error": str(e)}

    extra("C2 colVars", lambda: shard.colstats("var1", na_rm=True,
                                               out=col_out, warn=col_warn),
          "colVars")
    extra("C2 colMaxs", lambda: shard.colstats("max", na_rm=True), "colMaxs")
    extra("C2 rowMaxs", lambda: shard.rowstats("max", na_rm=True, group=grp),
          "rowSums")
    extra("C2 sum(svt)", lambda: shard.summarize("sum", na_rm=True),
          "colSums")
    extra("C2 var(svt)", lambda: shard.summarize("var1", na_rm=True),
          "colSums")
    # the atomic-free two-pass row kernels (north_star item 3) beside the
    # shared-memory histogram that runs by default
    old = env_set(SVTGPU_ROW_HIST="off")
    extra("C2 rowSums [atomic-free row_strips]", lambda: run_op("rowSums"),
          "rowSums")
    extra("C2 rowVars [atomic-free row_strips]", lambda: run_op("rowVars"),
          "rowVars")
    env_restore(old)
    try:   # rowsum() / colsum(): kernel time as the library reports it
        rng = np.random.Generator(np.random.PCG64(3))
        rg = rng.integers(1, 13, size=NROW).astype(np.int32)
        cg = rng.integers(1, 9, size=ncol).astype(np.int32)
        for name, fn in (("C2 rowsum(12 groups)",
                          lambda: shard.rowsum(rg, 12, na_rm=True)),
                         ("C2 colsum(8 groups)",
                          lambda: shard.colsum(cg, 8, na_rm=True))):
            fn()
            ms = min(fn()[2] for _ in range(3))
            per_op[name] = entry(ms, nnz, algorithmic_bytes("rowSums", nnz,
                                                            ncol, NROW), peak)
    except Exception as e:
        per_op["C2 rowsum/colsum"] = {"error": str(e)}

    # =====================================================================
    # CPU baseline (N = 1 only) and the in-bench parity check against it
    base = None
    parity = {"checked": False}
    cpu_outs = {}
    x_cpu = None
    if world == 1 and not args.no_cpu:
        try:
            base, c2_outs, x_cpu = cpu_c2(min(args.cpu_cols, ncol), 3)
            base.pop("ms_per_step", None)
        except Exception as e:   # the oracle always exists; say why if not
            base = {"value": None, "unit": "nnz/s", "cores": 0,
                    "kind": "reference", "sample": "failed: %s" % e}
        if x_cpu is not None:
            # the same kernels on the same columns: a view of the first
            # cpu_cols columns of the timed shard (the generator is
            # counter-based, so these are the reference sample's columns)
            sc = x_cpu.dim[1]
            view = DeviceSVT(NROW, sc, x_cpu.nnz, "integer",
                             shard.leaf_ptr[:sc + 1], shard.offs, shard.vals)
            worst = {}
            worst["colSums"] = _same("colSums", run_op("colSums", view,
                                                       None).cpu(),
                                     c2_outs[0])
            worst["colMeans"] = _same("colMeans", run_op("colMeans", view,
                                                         None).cpu(),
                                      c2_outs[1], rtol=1e-12)
            worst["rowSums"] = _same("rowSums", run_op("rowSums", view,
                                                       None).cpu(),
                                     c2_outs[2])
            worst["rowVars"] = _same("rowVars", run_op("rowVars", view,
                                                       None).cpu(),
                                     c2_outs[3], rtol=1e-12)
            # full-size outputs of the timed run: the first columns against
            # the reference, and size-independent identities for the rest
            cs = run_op("colSums").cpu().numpy().copy()
            _same("colSums[full][:sample]", cs[:sc], c2_outs[0])
            rs = run_op("rowSums").cpu().numpy()
            if float(cs.sum()) != float(rs.sum()):
                raise ParityError("sum(colSums) != sum(rowSums) at full size")
            mean_, var_ = shard.rowmoments(na_rm=True)
            cna = shard.rowstats("countNAs")[0].cpu().numpy()
            _same("rowMeans*nvals == rowSums",
                  mean_.cpu().numpy() * (ncol - cna), rs, rtol=1e-12)
            del view
            parity = {"checked": True,
                      "sample_vs_reference": "bit-exact colSums/rowSums, "
                      "<=1e-12 colMeans/rowVars on the first %d columns "
                      "(same kernels, same data)" % sc,
                      "full_size": "colSums[:sample] bit-exact vs reference; "
                                   "sum(colSums)==sum(rowSums); "
                                   "rowMeans*nvals==rowSums",
                      "worst_rel_err": worst}

    # =====================================================================
    # C3: SVT x dense products on the same matrix as double
    e2e_per = {}
    if not args.no_products:
        K = K_DENSE
        vals_d = shard.vals.to(torch.float64)
        vals_d[shard.vals == -2**31] = torch.tensor(
            [0x7FF00000000007A2], dtype=torch.int64,
            device=dev).view(torch.float64)[0]   # NA_real_
        dsh = DeviceSVT(NROW, ncol, nnz, "double", shard.leaf_ptr, shard.offs,
                        vals_d, leaf0=shard.leaf0,
                        nleaf_total=shard.nleaf_total)
        Yh, Dh = dense_operands(ncol)
        Y = torch.from_numpy(np.ascontiguousarray(Yh)).to(dev)   # row-major
        D = torch.from_numpy(np.ascontiguousarray(Dh)).to(dev)
        out_cp = torch.empty(ncol * K, dtype=torch.float64, device=dev)
        out_mm = torch.empty(NROW * K, dtype=torch.float64, device=dev)
        pb = product_bytes(nnz, ncol, NROW, K)
        # on-chip floor of the gather: K*8 B of the dense operand per nonzero
        # through shared memory at 128 B/clk/SM
        sm_floor_ms = nnz * (K * 8) / (128.0 * 148 * 1.965e9) * 1e3
        for name, fn in (
                ("C3 crossprod(svt, Y[33538x50])",
                 lambda: dsh.crossprod(Y, out=out_cp)),
                ("C3 svt %*% D[ncol x 50]",
                 lambda: dsh.matmul(D, group=grp, out=out_mm))):
            try:
                # first_call_ms includes the once-per-matrix work cached in
                # the handle (for %*% the device transpose)
                t_first = time.perf_counter()
                fn()
                barrier()
                t_first = (time.perf_counter() - t_first) * 1e3
                ms = dev_ms(fn, reps=5, warm=1)
                per_op[name] = entry(
                    ms, nnz, pb, peak,
                    GFLOPs_fp64=2 * K * nnz / (ms * 1e-3) / 1e9,
                    first_call_ms=round(t_first, 1),
                    frac_of_shared_memory_floor=sm_floor_ms / ms,
                    shared_memory_floor_ms=round(sm_floor_ms, 2))
            except Exception as e:
                per_op[name] = {"error": str(e)}
        if world > 1:   # the nrow x K allreduce of %*% alone
            try:
                ms = dev_ms(lambda: dist.all_reduce(out_mm), reps=10)
                per_op["C3 svt %%*%% D: allreduce of the partial products "
                       "(%.1f MB)" % (NROW * K * 8 / 1e6)] = \
                    {"ms": round(ms, 4)}
            except Exception as e:
                per_op["C3 %*% allreduce"] = {"error": str(e)}
        # double-input statistics on the same matrix (28.2 GB)
        st6 = torch.empty(6 * NROW, dtype=torch.float64, device=dev)
        for name, fn, key in (
                ("C2-as-double colSums",
                 lambda: dsh.colstats("sum", na_rm=True, out=col_out,
                                      warn=col_warn), "colSums"),
                ("C2-as-double colVars",
                 lambda: dsh.colstats("var1", na_rm=True, out=col_out,
                                      warn=col_warn), "colVars"),
                ("C2-as-double rowSums",
                 lambda: dsh.rowstats("sum", na_rm=True, group=grp,
                                      state=st3), "rowSums"),
                ("C2-as-double rowVars",
                 lambda: dsh.rowmoments(na_rm=True, group=grp, state=st6),
                 "rowVars")):
            try:
                ms = dev_ms(fn, reps=3, warm=1)
                per_op[name] = entry(ms, nnz, algorithmic_bytes(
                    key, nnz, ncol, NROW, vsz=8), peak)
            except Exception as e:
                per_op[name] = {"error": str(e)}
        del st6

    # =====================================================================
    # CPU legs of the other configurations + parity of the GPU on the same
    # inputs (N = 1)
    if world == 1 and x_cpu is not None:
        try:
            skip = set()
            if args.no_products:
                skip.add("C3")
            if args.no_configs:
                skip.update(("C1", "C5"))
            per_cfg, cpu_outs = cpu_other_configs(
                x_cpu, min(args.cpu_prod_cols, x_cpu.dim[1]),
                args.cpu_c5_cols, skip)
            try:
                from oracle import refcall as _rc
                per_cfg["sparse_crossprod_s (benchmark_crossprod.R shapes)"] \
                    = time_sparse_crossprod(_rc.crossprod1_SVT,
                                            _rc.crossprod2_SVT_SVT)
            except Exception as e:
                per_cfg["sparse_crossprod_s"] = {"error": str(e)}
            base["per_config"] = per_cfg
        except Exception as e:
            base["per_config"] = {"error": str(e)}
        if "crossprod" in cpu_outs and not args.no_products:
            pc = cpu_outs["c3_sample"].dim[1]
            e1 = cpu_outs["c3_sample"].nnz
            view = DeviceSVT(NROW, pc, e1, "double", shard.leaf_ptr[:pc + 1],
                             shard.offs, vals_d)
            Ys, Ds = dense_operands(pc)
            Yd = torch.from_numpy(np.ascontiguousarray(Ys)).to(dev)
            Dd = torch.from_numpy(np.ascontiguousarray(Ds)).to(dev)
            # The terms of a dot product are summed in a different order
            # than the reference's and can cancel (Y, D ~ N(0, 1)): the
            # bound is 1e-12 of sum |x||y| -- the condition of the dot
            # product -- computed with the same kernel on absolute values.
            va = torch.abs(torch.nan_to_num(vals_d[:e1]))
            aview = DeviceSVT(NROW, pc, e1, "double",
                              shard.leaf_ptr[:pc + 1], shard.offs, va)

            def prod_err(name, got, ref, cond):
                ref = np.asarray(ref)
                if not np.array_equal(np.isnan(got), np.isnan(ref)):
                    raise ParityError("%s: NA/NaN pattern differs" % name)
                m = ~np.isnan(ref)
                worst = float((np.abs(got[m] - ref[m]) /
                               np.maximum(cond[m], 1e-300)).max())
                if worst > 1e-12:
                    raise ParityError("%s: error %.3g of sum|x||y| > 1e-12"
                                      % (name, worst))
                return worst

            got = view.crossprod(Yd).cpu().numpy().reshape((pc, K_DENSE),
                                                           order="F")
            cond = aview.crossprod(torch.abs(Yd)).cpu().numpy().reshape(
                (pc, K_DENSE), order="F")
            parity["C3 crossprod err / sum|x||y|"] = prod_err(
                "crossprod", got, cpu_outs["crossprod"], cond)
            got = view.matmul(Dd).cpu().numpy().reshape((NROW, K_DENSE))
            cond = aview.matmul(torch.abs(Dd)).cpu().numpy().reshape(
                (NROW, K_DENSE))
            parity["C3 %*% err / sum|x||d|"] = prod_err(
                "%*%", got, cpu_outs["matmul"], cond)
            del view, aview, va, Yd, Dd
            cpu_outs["c3_sample"].release()

    # =====================================================================
    # end to end through the reference-facing API, host buffers
    e2e = None
    if not args.no_e2e:
        # the host copy of the matrix is split over the ranks (the box has
        # one host memory: 18.8 GB per 1e6 columns)
        ecols = args.e2e_cols or max(1, ncol // world)
        ptr = shard.leaf_ptr[:ecols + 1].cpu().numpy()
        ennz = int(ptr[-1])
        offs = shard.offs[:ennz].cpu().numpy()
        vals = shard.vals[:ennz].cpu().numpy()
        hx = SVT_SparseArray((NROW, ecols), "integer", ptr, offs, vals)
        hx.r_SVT
        # same thread-control setting as the reference arm: all host cores
        # (they only drive the host-side flatten here)
        sa.set_SparseArray_nthread(max(1, (os.cpu_count() or 1) // world))

        def stock_calls():
            sharded.colSums(hx, na_rm=True)
            sharded.colMeans(hx, na_rm=True)
            sharded.rowSums(hx, na_rm=True, group=group_cpu)
            sharded.rowVars(hx, na_rm=True, group=group_cpu)

        def e2e_step():
            # options(SparseArray.gpu.cache = TRUE): the device CSC of the
            # SVT is kept between consecutive .Calls on the same object
            # (fingerprint over all leaves checked on every call).  The
            # cache is dropped at the start of every step, so every step
            # pays its own flatten + upload from host memory.
            sa.set_gpu_cache(None)
            stock_calls()

        def timed(step, steps):
            step()
            barrier()
            tot0 = dict(rcall.totals)
            t0 = time.perf_counter()
            for _ in range(steps):
                step()
            barrier()
            dt = maxr((time.perf_counter() - t0) / steps)
            return dt, {k: (rcall.totals[k] - tot0[k]) / steps
                        for k in ("h2d_bytes", "d2h_bytes", "calls")}

        ennz_all = sumr(ennz)
        # stateless first (no cache: every call flattens + uploads)
        sa.set_gpu_cache(False)
        dt0, tot0_ = timed(stock_calls, args.e2e_steps)
        last0 = rcall.last_timings()
        sa.set_gpu_cache(True)
        dt, tot = timed(e2e_step, args.e2e_steps)
        sa.set_gpu_cache(False)
        e2e = {"value": len(OPS) * ennz_all / dt, "unit": "nnz/s",
               "h2d_bytes_per_step": int(tot["h2d_bytes"]),
               "d2h_bytes_per_step": int(tot["d2h_bytes"]),
               "ms_per_step": dt * 1e3, "steps": args.e2e_steps,
               "cols_per_gpu": ecols, "calls_per_step": int(tot["calls"]),
               "api": "colSums/colMeans/rowSums/rowVars(svt, na.rm=TRUE) "
                      "through the unchanged .Call entry points "
                      "(C_colStats_SVT x2, C_rowStats_SVT x4: rowVars is "
                      "countNAs + sum + centered_X2_sum as in the R method) "
                      "on a HOST SVT with options(SparseArray.gpu.cache=TRUE):"
                      " the first call of a step flattens the leaves and "
                      "uploads them through pinned staging (uint16 offsets / "
                      "int8 values when they fit); the other five find the "
                      "same object by its leaf fingerprint and reuse the "
                      "device CSC.  The cache is dropped at the start of "
                      "every timed step.",
               "no_cache": {
                   "value": len(OPS) * ennz_all / dt0, "unit": "nnz/s",
                   "ms_per_step": dt0 * 1e3,
                   "h2d_bytes_per_step": int(tot0_["h2d_bytes"]),
                   "calls_per_step": int(tot0_["calls"]),
                   "api": "the same step stateless (cache off, the default): "
                          "every one of the 6 calls flattens + uploads",
                   "last_call_phases_ms": {k: round(v, 3)
                                           for k, v in last0.items()
                                           if k.endswith("_ms")}}}

        # the same step with the one-pass C_rowMoments_SVT patch of
        # INTEGRATION.md (rowVars = ONE call instead of three)
        def onepass_step():   # stateless (cache off)
            sharded.colSums(hx, na_rm=True)
            sharded.colMeans(hx, na_rm=True)
            sharded.rowSums(hx, na_rm=True, group=group_cpu)
            sa.rowMoments(hx, na_rm=True)

        try:
            if world > 1:
                raise RuntimeError("single-GPU key (shards would need the "
                                   "raw moments, not mean / var)")
            dt1, tot1 = timed(onepass_step, args.e2e_steps)
            e2e["onepass_rowVars"] = {
                "value": len(OPS) * ennz_all / dt1, "unit": "nnz/s",
                "ms_per_step": dt1 * 1e3,
                "h2d_bytes_per_step": int(tot1["h2d_bytes"]),
                "calls_per_step": int(tot1["calls"]),
                "api": "same step, rowVars through the one-pass "
                       "C_rowMoments_SVT entry point (INTEGRATION.md patch "
                       "of the R method): 4 uploads instead of 6"}
        except Exception as e:
            e2e["onepass_rowVars"] = {"error": str(e)}

        # the same step with the matrix made device-resident first: ONE
        # flatten + upload per step (inside the timed region), then the same
        # six .Call's on the handle (INTEGRATION.md: C_svtgpu_resident_SVT)
        def resident_step():
            r = sa.to_device(hx)
            sharded.colSums(r, na_rm=True)
            sharded.colMeans(r, na_rm=True)
            sharded.rowSums(r, na_rm=True, group=group_cpu)
            sharded.rowVars(r, na_rm=True, group=group_cpu)
            r.release()

        dtr, totr = timed(resident_step, args.e2e_steps)
        e2e["resident"] = {
            "value": len(OPS) * ennz_all / dtr, "unit": "nnz/s",
            "ms_per_step": dtr * 1e3,
            "h2d_bytes_per_step": int(totr["h2d_bytes"]),
            "d2h_bytes_per_step": int(totr["d2h_bytes"]),
            "api": "to_device(svt) once per step (flatten + upload, timed), "
                   "then the same calls on the resident handle"}

        # host copy bandwidth of this box, same run: what the flatten (a
        # gather of the leaves into pinned slots) competes with
        try:
            nthr = max(1, (os.cpu_count() or 1) // world)
            e2e["host_memcpy_GBps"] = round(host_copy_bandwidth(
                min(ennz * 4, 1 << 31), nthr), 1)
            e2e["host_memcpy_note"] = ("numpy copies of %d slices on %d "
                                       "threads, read + written bytes"
                                       % (nthr, nthr))
        except Exception as e:
            e2e["host_memcpy_GBps"] = "n/a: %s" % e

        # ---- C3 end to end: crossprod(svt, Y) / svt %*% D from host --------
        if not args.no_products and world == 1:
            try:
                hxd = hx.with_type("double")
                hx.release()
                hxd.r_SVT
                Yh, Dh = dense_operands(ecols)
                for name, fn in (
                        ("C3 crossprod(svt, Y[33538x50])",
                         lambda: sa.crossprod(hxd, Yh)),
                        ("C3 svt %*% D[ncol x 50]",
                         lambda: sa.matmul(hxd, Dh))):
                    tot0 = dict(rcall.totals)
                    t = best_wall(fn, n=2, warm=1)
                    e2e_per[name] = {
                        "value": ennz / t, "unit": "nnz/s",
                        "seconds": round(t, 4),
                        "h2d_bytes_per_call": int(
                            (rcall.totals["h2d_bytes"] - tot0["h2d_bytes"])
                            / 3),
                        "d2h_bytes_per_call": int(
                            (rcall.totals["d2h_bytes"] - tot0["d2h_bytes"])
                            / 3),
                        "phases_ms": {k: round(v, 2) for k, v in
                                      rcall.last_timings().items()
                                      if k.endswith("_ms")}}
                hxd.release()
                del hxd
            except Exception as e:
                e2e_per["C3"] = {"error": str(e)}
        else:
            hx.release()
        del hx

    if not args.no_products:
        del dsh, vals_d, Y, D, out_cp, out_mm
    torch.cuda.empty_cache()

    # =====================================================================
    # C1 and C5 (N = 1): kernels device-resident, end to end from host,
    # parity against the reference's outputs on the same inputs
    if world == 1 and not args.no_configs:
        try:
            from sparsearray_b200 import synth
            x1 = cpu_outs.get("c1_matrix") or synth.random_svt(
                C1_DIM[0], C1_DIM[1], C1_DENSITY, seed=1)
            x1.r_SVT
            d1 = DeviceSVT.from_host(x1)
            c1_e2e = {}
            absv = np.abs(x1.vals)
            c1_cond = {"colSums": np.add.reduceat(
                           np.append(absv, 0.0),
                           np.minimum(x1.ptr[:-1], absv.size)) *
                       (np.diff(x1.ptr) > 0),
                       "rowSums": np.bincount(x1.offs, weights=absv,
                                              minlength=C1_DIM[0])}
            for name, kfn, efn, key in (
                    ("colSums", lambda: d1.colstats("sum"),
                     lambda: sa.colSums(x1), "colSums"),
                    ("colVars", lambda: d1.colstats("var1"),
                     lambda: sa.colVars(x1), "colVars"),
                    ("rowSums", lambda: d1.rowstats("sum"),
                     lambda: sa.rowSums(x1), "rowSums"),
                    ("rowVars", lambda: d1.rowmoments()[1],
                     lambda: sa.rowVars(x1), "rowVars")):
                ms = dev_ms(kfn, reps=20, warm=3)
                per_op["C1 " + name] = entry(
                    ms, x1.nnz, algorithmic_bytes(key, x1.nnz, C1_DIM[1],
                                                  C1_DIM[0], vsz=8), peak,
                    note="launch-bound: 60 MB is ~10 us of HBM time")
                c1_e2e[name] = {"ms": round(best_wall(efn, n=7) * 1e3, 4)}
                if "C1 " + name in cpu_outs:
                    parity["C1 " + name] = _same(
                        "C1 " + name, np.asarray(efn()),
                        cpu_outs["C1 " + name], rtol=1e-12,
                        cond=c1_cond.get(name))
            rx = sa.to_device(x1)
            for name, efn in (("colSums", lambda: sa.colSums(rx)),
                              ("colVars", lambda: sa.colVars(rx)),
                              ("rowSums", lambda: sa.rowSums(rx)),
                              ("rowVars", lambda: sa.rowVars(rx))):
                c1_e2e[name]["resident_ms"] = round(
                    best_wall(efn, n=7) * 1e3, 4)
            rx.release()
            e2e_per["C1 20000x5000 double d=0.05 (nnz=%d)" % x1.nnz] = {
                "ops": c1_e2e,
                "api": "sa.colSums/colVars/rowSums/rowVars(host SVT) through "
                       ".Call, best of 7; resident_ms = the same calls on a "
                       "to_device() handle"}
            d1.free()
            x1.release()
        except ParityError:
            raise
        except Exception as e:
            per_op["C1"] = {"error": str(e)}

        try:
            c5n = args.c5_cols
            l5 = DeviceSVT.generate_poisson(C5_NROW, c5n, C5_DENSITY, seed=5,
                                            lacunar=True)
            n5 = l5.nnz
            rng = np.random.Generator(np.random.PCG64(3))
            rg5 = rng.integers(1, 13, size=C5_NROW).astype(np.int32)
            cg5 = rng.integers(1, 9, size=c5n).astype(np.int32)
            for name, fn, key in (
                    ("colSums", lambda: l5.colstats("sum"), "colSums"),
                    ("rowSums", lambda: l5.rowstats("sum"), "rowSums"),
                    ("rowVars", lambda: l5.rowmoments()[1], "rowVars"),
                    ("rowMaxs", lambda: l5.rowstats("max"), "rowSums")):
                ms = dev_ms(fn, reps=5)
                per_op["C5 " + name] = entry(
                    ms, n5, algorithmic_bytes(key, n5, c5n, C5_NROW, vsz=0),
                    peak)
            for name, fn in (("rowsum(12 groups)",
                              lambda: l5.rowsum(rg5, 12)),
                             ("colsum(8 groups)",
                              lambda: l5.colsum(cg5, 8))):
                fn()
                ms = min(fn()[2] for _ in range(3))
                per_op["C5 " + name] = entry(
                    ms, n5, algorithmic_bytes("rowSums", n5, c5n, C5_NROW,
                                              vsz=0), peak)
            if "c5_sample" in cpu_outs:
                x5 = cpu_outs["c5_sample"]
                sc = x5.dim[1]
                v5 = DeviceSVT(C5_NROW, sc, x5.nnz, "integer",
                               l5.leaf_ptr[:sc + 1], l5.offs, None)
                parity["C5 colSums"] = _same(
                    "C5 colSums", v5.colstats("sum")[0].cpu(),
                    cpu_outs["C5 colSums"])
                parity["C5 rowSums"] = _same(
                    "C5 rowSums", v5.rowstats("sum")[0].cpu(),
                    cpu_outs["C5 rowSums"])
                parity["C5 rowVars"] = _same(
                    "C5 rowVars", v5.rowmoments()[1].cpu(),
                    cpu_outs["C5 rowVars"], rtol=1e-12)
                del v5
                x5.release()
            # end to end from a host lacunar SVT (offsets only: 8 GB)
            if not args.no_e2e:
                ptr5 = l5.leaf_ptr.cpu().numpy()
                offs5 = l5.offs[:n5].cpu().numpy()
                h5 = SVT_SparseArray((C5_NROW, c5n), "integer", ptr5, offs5,
                                     None)
                h5.r_SVT
                c5_e2e = {}
                for name, fn in (("colSums", lambda: sa.colSums(h5)),
                                 ("rowSums", lambda: sa.rowSums(h5)),
                                 ("rowVars", lambda: sa.rowVars(h5))):
                    t = best_wall(fn, n=2, warm=1)
                    c5_e2e[name] = {"ms": round(t * 1e3, 2),
                                    "nnz_per_s": n5 / t}
                e2e_per["C5 lacunar %d x %d d=0.01 (nnz=%d)"
                        % (C5_NROW, c5n, n5)] = {
                    "ops": c5_e2e, "api": "sa.colSums/rowSums/rowVars(host "
                                          "lacunar SVT) through .Call"}
                h5.release()
                del h5, ptr5, offs5
            l5.free()
            del l5
        except ParityError:
            raise
        except Exception as e:
            per_op["C5"] = {"error": str(e)}
    if x_cpu is not None:
        x_cpu.release()
    torch.cuda.empty_cache()

    # =====================================================================
    # C4 as written: ONE 33,538 x 4,000,000 matrix, column-sharded over the
    # ranks (strong scaling); rowSums + rowVars with the allreduce
    strong = None
    if not args.no_configs:
        try:
            del shard
            torch.cuda.empty_cache()
            c4 = args.c4_cols
            lo, hi = (c4 * rank) // world, (c4 * (rank + 1)) // world
            sh4 = DeviceSVT.generate_poisson(
                NROW, hi - lo, DENSITY, seed=4, na_rate=NA_RATE, leaf0=lo,
                nleaf_total=c4)
            nnz4 = sumr(sh4.nnz)

            def c4_step():
                sh4.rowstats("sum", na_rm=True, group=grp, state=st3)
                sh4.rowmoments(na_rm=True, group=grp, state=st4)

            k4 = max(3, min(args.steps, 20))
            ms = maxr(dev_ms(c4_step, reps=k4, warm=3))
            b4 = 2 * (nnz4 * 8 + (c4 + 1) * 8)
            strong = {"workload": "configs[3]: 33538 x %d int counts d=0.07 "
                                  "(nnz=%d) column-sharded over %d GPU(s); "
                                  "step = rowSums + rowVars (na.rm=TRUE) "
                                  "with the NCCL allreduce of the row states"
                                  % (c4, int(nnz4), world),
                      "scaling": "strong", "n_gpus": world,
                      "ms_per_step": round(ms, 4), "steps": k4,
                      "value": 2 * nnz4 / (ms * 1e-3), "unit": "nnz/s",
                      "GBps_aggregate": b4 / (ms * 1e-3) / 1e9,
                      "frac_of_aggregate_hbm_peak":
                          b4 / (ms * 1e-3) / 1e9 / (peak * world)}
            sh4.free()
            del sh4
        except Exception as e:
            strong = {"error": str(e)}

    roofline["per_op"] = per_op
    if strong is not None:
        roofline["strong_scaling_c4"] = strong
    if e2e is not None:
        e2e["per_config"] = e2e_per

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "nnz/s",
            "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32->f64",
            "data": "synthetic",
            "config": {
                "workload": "configs[1]: 33538x%d int counts d=0.07 per GPU "
                            "(nnz=%d), colSums/colMeans/rowSums/rowVars "
                            "na.rm=TRUE" % (ncol, nnz),
                "l2": "inputs (%.1f GB per GPU) larger than L2, no flush"
                      % ((nnz * 8) / 1e9),
                "sharding": "columns; rowSums/rowVars states allreduced "
                            "(NCCL)" if world > 1 else "single GPU",
                "warmup_note": "warm-up forced to >= %d steps (nvidia-smi "
                               "start-up + clock sampling under load); "
                               "--warmup %d was requested"
                               % (MIN_WARMUP, args.warmup),
                "parity_checked": parity},
            "roofline": roofline, "cpu_baseline": base, "e2e": e2e,
            "gpu_launches": int(launches), "clocks": clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
