// Quasi-Newton Hessians of the lock-step interior-point driver (dnlp_b200/lockstep_ipm.py, hessian_approximation =
// "limited-memory"): one dense damped-BFGS matrix W_b (n x n, symmetric) per start, the update of the test-suite's
// serial stand-in (tests/cyipopt_standin.py) applied to a list of starts at once.
//
// Storage: the lower triangle of W_b, packed and batch fastest like every output of the batched engine: entry
// (i, j <= i) at p = i (i + 1) / 2 + j, start b at Wq[p * B + b].  Bitwise symmetry is then a property of the layout.
//
// The update of one start (s, y: the step and the change of the Lagrangian's gradient):
//   Bs_i = sum_j W_ij s_j                      (j = 0 .. n-1 in order)
//   sBs  = sum_i s_i Bs_i,  sy = sum_i s_i y_i (i = 0 .. n-1 in order)
//   skip the start unless sBs > 0             (NaN, 0 or negative: W_b untouched, applied = 0)
//   theta = 1 if sy >= 0.2 sBs else 0.8 sBs / (sBs - sy)
//   r_i  = theta y_i + (1 - theta) Bs_i,  sr = sum_i s_i r_i
//   W_ij := (W_ij - (Bs_i Bs_j) / sBs) + (r_i r_j) / sr
// Every per-start quantity is computed by one thread in a fixed order from that start's data only, so a start's
// result does not depend on which other starts are in the call.  The vectors of the selected starts live in
// n x count scratch arrays, start fastest, so that the GEMV and the rank-2 update read them coalesced next to W.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace dnlp_qn {

// row i of packed entry p: the largest i with i (i + 1) / 2 <= p
__device__ inline int64_t packed_row(int64_t p) {
  int64_t i = (int64_t)((sqrt(8.0 * (double)p + 1.0) - 1.0) * 0.5);
  while (i * (i + 1) / 2 > p) --i;
  while ((i + 1) * (i + 2) / 2 <= p) ++i;
  return i;
}

// W_b := I for every start b
__global__ void qn_identity_kernel(double *Wq, int64_t np, int B) {
  const int64_t total = np * B;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = e / B, i = packed_row(p);
    Wq[e] = p - i * (i + 1) / 2 == i ? 1.0 : 0.0;
  }
}

// S, Y (count x n, start-major, as copied in) -> St, Yt (n x count, start fastest)
__global__ void qn_transpose_kernel(const double *__restrict__ S, const double *__restrict__ Y, double *St, double *Yt,
                                    int64_t n, int count) {
  const int64_t total = n * count;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = e / count, c = e - j * count;
    St[e] = S[c * n + j];
    Yt[e] = Y[c * n + j];
  }
}

// Bs[i, c] = sum_j W_ij s_j in the order j = 0 .. n-1: one thread per (row, selected start), start fastest, so the
// reads of W (row i: packed entries i(i+1)/2 .. i(i+1)/2 + i, then column i below the diagonal) coalesce over starts
__global__ void qn_gemv_kernel(const double *__restrict__ Wq, int B, const int32_t *__restrict__ starts, int count,
                               const double *__restrict__ St, double *Bs, int64_t n) {
  const int64_t total = n * count;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / count, c = e - i * count;
    const double *w = Wq + starts[c];
    const double *s = St + c;
    double acc = 0.0;
    const int64_t row = i * (i + 1) / 2;
    for (int64_t j = 0; j < i; ++j) acc += w[(row + j) * B] * s[j * count];
    for (int64_t j = i, p = row + i; j < n; ++j, p += j) acc += w[p * B] * s[j * count];
    Bs[e] = acc;
  }
}

// One thread per selected start: sBs, sy, theta, r (into R) and sr, each sum in the order i = 0 .. n-1.
// coef[c] = sBs, coef[count + c] = sr; applied[c] = 1 when the start is updated.
__global__ void qn_coef_kernel(const double *__restrict__ St, const double *__restrict__ Yt,
                               const double *__restrict__ Bs, double *R, double *coef, int32_t *applied, int64_t n,
                               int count) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= count) return;
  double sBs = 0.0, sy = 0.0;
  for (int64_t i = 0; i < n; ++i) {
    const double s = St[i * count + c];
    sBs += s * Bs[i * count + c];
    sy += s * Yt[i * count + c];
  }
  const bool ok = sBs > 0.0;           // false for NaN too
  const double theta = sy >= 0.2 * sBs ? 1.0 : 0.8 * sBs / (sBs - sy);
  double sr = 0.0;
  if (ok)
    for (int64_t i = 0; i < n; ++i) {
      const double r = theta * Yt[i * count + c] + (1.0 - theta) * Bs[i * count + c];
      R[i * count + c] = r;
      sr += St[i * count + c] * r;
    }
  coef[c] = sBs;
  coef[count + c] = sr;
  applied[c] = ok ? 1 : 0;
}

// One thread per (packed entry, selected start), start fastest: W_ij := (W_ij - (Bs_i Bs_j) / sBs) + (r_i r_j) / sr
__global__ void qn_rank2_kernel(double *Wq, int B, const int32_t *__restrict__ starts, int count,
                                const double *__restrict__ Bs, const double *__restrict__ R,
                                const double *__restrict__ coef, const int32_t *__restrict__ applied, int64_t np) {
  const int64_t total = np * count;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = e / count, c = e - p * count;
    if (!applied[c]) continue;
    const int64_t i = packed_row(p), j = p - i * (i + 1) / 2;
    const double sBs = coef[c], sr = coef[count + c];
    const double bi = Bs[i * count + c], bj = Bs[j * count + c];
    const double ri = R[i * count + c], rj = R[j * count + c];
    double *w = Wq + p * B + starts[c];
    *w = (*w - (bi * bj) / sBs) + (ri * rj) / sr;
  }
}

}  // namespace dnlp_qn
