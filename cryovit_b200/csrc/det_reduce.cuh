// Deterministic mode of head training: the pieces every fixed-order reduction shares.
//
// A reduction that the default kernels finish with float atomics (shared-memory and global atomicAdd, red.global.add)
// runs in deterministic mode as
//   1. the same kernel body, each block (or CTA) writing its partial result as one row of a caller-owned scratch slab
//      [rows][n] with plain stores, its in-block sums taken in a fixed thread order, and
//   2. det_finalize: out[j] (=|+=) sum over r = 0 .. rows - 1 of partials[r][j], in an order that depends on rows and
//      n only.
// rows is a function of the problem shape and the SM count, never of which block finishes first, so a run on the same
// GPU gives bit-identical results.
#pragma once
#include "tmap.h"

namespace cvit {

// out[j] = (add ? out[j] : 0) + sum_r partials[r * ld + j] for j < n (ld = n: a dense [rows][n] slab): fp64, rows
// r = ry, ry + 8, ... in order per lane ry, the eight lanes added 0 .. 7. rows >= 1.
int det_finalize(const float* partials, int64_t rows, int64_t n, int64_t ld, float* out, bool add, cudaStream_t stream);

// The fp64 [rows][8] variant: cvit_conv3d_rows8_score's finalize (csrc/conv_rows8.cu), out8 overwritten.
int rows8_score_finalize(const double* partials, int rows, double* out8, cudaStream_t stream);

// In-block fixed-order column sums. Thread t of the block has 8 partial sums sh[t * 8 + k] for channels vec(t) * 8 + k,
// vec(t) = (t + phase) % nvec; threads t >= tn hold nothing. row[c] = sum over t = t0(c), t0(c) + nvec, ... < tn of
// sh[t * 8 + c % 8] (t increasing). Call after __syncthreads(); every thread of the block takes part.
__device__ __forceinline__ void det_block_colsum(const float* sh, int C, int nvec, int tn, int phase, float* __restrict__ row) {
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int v = c >> 3, k = c & 7;
    float s = 0.f;
    for (int t = ((v - phase) % nvec + nvec) % nvec; t < tn; t += nvec) s += sh[t * 8 + k];
    row[c] = s;
  }
}

// Scratch check shared by the *_det entry points: a null scratch or fewer than `need` elements is refused before any
// launch.
inline int det_check_scratch(const void* scratch, int64_t have, int64_t need, const char* what) {
  if (!scratch || have < need) {
    set_error("%s: scratch of %lld elements needed, got %lld%s", what, (long long)need, (long long)have, scratch ? "" : " (null)");
    return CVIT_ERR_INVALID;
  }
  return CVIT_OK;
}

}  // namespace cvit
