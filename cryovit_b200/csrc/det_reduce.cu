// The one finalize kernel of deterministic mode (see det_reduce.cuh): fixed-order sums of per-block partial rows.
#include "det_reduce.cuh"

namespace cvit {

// Block = 32 columns x 8 row lanes. Lane ry adds rows ry, ry + 8, ... in fp64; lane 0 then adds the eight lane sums in
// lane order. Reads are 128-byte coalesced per (row, 32 columns).
__global__ void __launch_bounds__(256) det_finalize_kernel(const float* __restrict__ partials, int64_t rows, int64_t n,
                                                           int64_t ld, float* __restrict__ out, int add) {
  __shared__ double red[8][32];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int64_t j = (int64_t)blockIdx.x * 32 + cx;
  double s = 0.0;
  if (j < n)
    for (int64_t r = ry; r < rows; r += 8) s += (double)partials[r * ld + j];
  red[ry][cx] = s;
  __syncthreads();
  if (ry == 0 && j < n) {
    double t = add ? (double)out[j] : 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][cx];
    out[j] = (float)t;
  }
}

int det_finalize(const float* partials, int64_t rows, int64_t n, int64_t ld, float* out, bool add, cudaStream_t stream) {
  det_finalize_kernel<<<(unsigned)((n + 31) / 32), 256, 0, stream>>>(partials, rows, n, ld, out, add ? 1 : 0);
  return check_launch("det_finalize_kernel");
}

}  // namespace cvit
