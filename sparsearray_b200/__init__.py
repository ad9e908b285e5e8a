"""sparsearray_b200 -- B200-native compute path for Bioconductor SparseArray's
SVT_SparseMatrix column/row statistics and SVT x dense products.

  svt      host-side mirror of the reference's R interface (drop-in calls
           through the unchanged .Call entry points, served by CUDA)
  device   device-resident column shards + multi-GPU composition
  synth    synthetic inputs with the reference generators' distributions
  _native  ctypes binding of the C ABI (include/svtgpu.h)
  build    in-tree build of libsvtgpu.so / libsvt_rglue.so

Importing the package never touches CUDA; the first call does, and fails
loudly when the extension or a device is missing (there is no CPU fallback).
"""
from .svt import (SVT_SparseArray, SVT_SparseMatrix, ResidentSVT, to_device,  # noqa: F401
                  from_csc, to_csc, Arith, Math, sweep, Compare, Logic,
                  is_na, is_nan, is_infinite, subset,
                  RArray, NA_INTEGER,
                  NA_REAL, is_na_real,
                  colSums, colMeans, colVars, colSds, colMins, colMaxs,
                  colRanges, colProds, colAnyNAs, colCountNAs, colAnys,
                  colAlls, colSums2, colMeans2, colMedians, rowMedians,
                  rowSums, rowMeans, rowVars, rowSds, rowMins, rowMaxs,
                  rowRanges, rowAnyNAs, rowCountNAs, rowSums2, rowMoments,
                  rowProds, rowMeans2, rowAnys, rowAlls,
                  crossprod, matmul, tcrossprod,
                  summarize_SVT, anyNA, svt_any, svt_all, svt_min, svt_max,
                  svt_range, svt_sum, svt_prod, mean, var, sd, rowsum, colsum)
from .rcall import (get_SparseArray_nthread, set_SparseArray_nthread,  # noqa: F401
                    last_timings, set_gpu_cache, gpu_cache_stats)
