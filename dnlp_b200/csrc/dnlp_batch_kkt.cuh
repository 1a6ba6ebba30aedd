// Batched KKT systems of the lock-step interior-point driver (dnlp_b200/lockstep_ipm.py), one dense system per start:
//
//   K_b = [[ W_b + diag(Sigma_b) + dw_b I ,  A_b' ],     W_b: Hessian of the Lagrangian in z = (x, slacks), from output HESS
//          [ A_b                          , -dc_b I ]]   A_b = [J_b, -P], J_b from output JAC, P selects the inequality rows
//
// Storage: K_b is M x M row-major (M = N + m) in a per-start slot of the workspace.  Assembly writes the full symmetric
// matrix; the factorisation overwrites the lower triangle with L (unit, implied) and D (on the diagonal) and never touches
// the strict upper triangle, so the upper triangle plus the saved diagonal remain the assembled K for the refinement
// step and for dnlp_batch_kkt_matrix.
//
// LDL' without pivoting, in the fixed order [x / slack block, constraint block].  By Sylvester's law the signs of D
// are the inertia of K whenever the factorisation completes.  A pivot d_j counts as zero when it is within 1e-11 of
// its own scale |K_jj| + sum_k L_jk^2 |d_k| (the terms whose sum it is cancelled).  A threshold relative to max|d|
// would not do here: without pivoting the constraint-block pivots are Schur complements of size a^2 / Sigma, many
// orders below the x-block pivots once Sigma spans 1e-12 .. 1e11, and raising dw only makes them smaller.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dnlp_kkt {

constexpr int NB = 32;        // panel width of the blocked factorisation
constexpr int TT = 64;        // trailing-update tile (TT x TT entries, 4 x 4 per thread)
constexpr int THREADS = 256;

// K of every selected start := 0 (slots are indexed by start id)
__global__ void kkt_zero_kernel(double *K, const int32_t *starts, int count, int64_t MM) {
  const int64_t total = (int64_t)count * MM;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = e / MM;
    K[(int64_t)starts[c] * MM + (e - c * MM)] = 0.0;
  }
}

// One thread per (target entry, selected start), start fastest: the output reads (len x B, batch fastest) coalesce.
// Target t sums its sources in the fixed order of src[sp[t] .. sp[t+1]): id < nnzH -> HESS[id], id >= nnzH ->
// JAC[id - nnzH], id == -1 -> the constant -1 of the slack column.  A diagonal target of the x / slack block then adds
// Sigma and dw, one of the constraint block is -dc:  K_ii = (W_ii + Sigma_i) + dw.
__global__ void kkt_scatter_kernel(double *K, double *Dg, double *Wd, const double *__restrict__ jac,
                                   const double *__restrict__ hess, int B, const int32_t *__restrict__ ti,
                                   const int32_t *__restrict__ tj, const int32_t *__restrict__ sp,
                                   const int32_t *__restrict__ src, int64_t ntgt, int64_t nnzH,
                                   const int32_t *__restrict__ starts, int count, const double *__restrict__ sigma,
                                   const double *__restrict__ dw, const double *__restrict__ dc, int64_t N, int64_t M) {
  const int64_t total = ntgt * count;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = e / count;
    const int c = (int)(e - t * count);
    const int64_t b = starts[c];
    double v = 0.0;
    for (int s = sp[t]; s < sp[t + 1]; ++s) {
      const int32_t id = src[s];
      v += id < 0 ? -1.0 : (id < nnzH ? hess[(int64_t)id * B + b] : jac[(int64_t)(id - nnzH) * B + b]);
    }
    const int64_t i = ti[t], j = tj[t];
    double *Kb = K + b * M * M;
    if (i == j) {
      if (i < N) {
        Wd[b * N + i] = v;
        v = (v + sigma[(int64_t)c * N + i]) + dw[c];
      } else {
        v = -dc[c];
      }
      Dg[b * M + i] = v;
      Kb[i * M + i] = v;
    } else {
      Kb[i * M + j] = v;
      Kb[j * M + i] = v;
    }
  }
}

__device__ inline double block_reduce(double v, bool is_max, double *red) {
  for (int o = 16; o > 0; o >>= 1) {
    const double w = __shfl_xor_sync(0xffffffffu, v, o);
    v = is_max ? fmax(v, w) : v + w;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  v = red[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) v = is_max ? fmax(v, red[w]) : v + red[w];
  return v;
}

// One CTA per selected start: blocked right-looking LDL' of the lower triangle, in place.  work: M doubles per
// selected start for the pivot scales.
__global__ void __launch_bounds__(THREADS) kkt_ldl_kernel(double *K, const int32_t *starts, int64_t M,
                                                          int32_t *inertia, double *work, int64_t work_stride) {
  __shared__ double Dblk[NB][NB + 1];
  __shared__ double Li[NB][TT + 1];      // panel rows of tile i, transposed (padded: the transposing stores spread over banks)
  __shared__ double Wj[NB][TT + 1];      // panel rows of tile j times D, transposed
  __shared__ double red[THREADS / 32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double *A = K + (int64_t)starts[blockIdx.x] * M * M;
  double *scale = work + blockIdx.x * work_stride;
  for (int64_t i = tid; i < M; i += THREADS) scale[i] = fabs(A[i * M + i]);
  __syncthreads();

  for (int64_t k0 = 0; k0 < M; k0 += NB) {
    const int kb = (int)(M - k0 < NB ? M - k0 : NB);
    // 1. the diagonal block: unblocked LDL' by one warp (lane = row)
    for (int idx = tid; idx < kb * kb; idx += THREADS) {
      const int r = idx / kb, c = idx - r * kb;
      if (c <= r) Dblk[r][c] = A[(k0 + r) * M + k0 + c];
    }
    __syncthreads();
    if (warp == 0) {
      const int r = lane;
      double sc = r < kb ? scale[k0 + r] : 0.0;
      for (int j = 0; j < kb; ++j) {
        const double d = Dblk[j][j];
        double l = 0.0;
        if (r > j && r < kb) {
          l = Dblk[r][j] / d;
          sc += l * l * fabs(d);
        }
        __syncwarp();
        if (r > j && r < kb) Dblk[r][j] = l;
        __syncwarp();
        if (r > j && r < kb)
          for (int c = j + 1; c <= r; ++c) Dblk[r][c] -= l * d * Dblk[c][j];
        __syncwarp();
      }
      if (r < kb) scale[k0 + r] = sc;
    }
    __syncthreads();
    for (int idx = tid; idx < kb * kb; idx += THREADS) {
      const int r = idx / kb, c = idx - r * kb;
      if (c <= r) A[(k0 + r) * M + k0 + c] = Dblk[r][c];
    }
    const int64_t k1 = k0 + kb;
    // 2. the panel below: W21 L11' = A21 (row by row), L21 = W21 D1^-1
    for (int64_t i = k1 + tid; i < M; i += THREADS) {      // in place: a thread's kb entries stay in L1
      double *row = A + i * M + k0;
      for (int j = 1; j < kb; ++j) {
        double s = row[j];
        for (int c = 0; c < j; ++c) s -= row[c] * Dblk[j][c];
        row[j] = s;
      }
      double sc = scale[i];
      for (int j = 0; j < kb; ++j) {
        const double l = row[j] / Dblk[j][j];
        row[j] = l;
        sc += l * l * fabs(Dblk[j][j]);
      }
      scale[i] = sc;
    }
    __syncthreads();
    // 3. trailing update of the lower triangle: A22 -= L21 D1 L21'
    const int64_t R = M - k1;
    const int nt = (int)((R + TT - 1) / TT);
    const int ty = tid >> 4, tx = tid & 15;
    for (int tjj = 0; tjj < nt; ++tjj) {
      for (int tii = tjj; tii < nt; ++tii) {
        const int64_t i0 = k1 + (int64_t)tii * TT, j0 = k1 + (int64_t)tjj * TT;
        for (int idx = tid; idx < NB * TT; idx += THREADS) {
          const int r = idx / NB, p = idx - r * NB;       // consecutive threads walk along a row
          const bool okp = p < kb;
          Li[p][r] = (okp && i0 + r < M) ? A[(i0 + r) * M + k0 + p] : 0.0;
          Wj[p][r] = (okp && j0 + r < M) ? A[(j0 + r) * M + k0 + p] * Dblk[p][p] : 0.0;
        }
        __syncthreads();
        double acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[a][q] = 0.0;
        for (int p = 0; p < kb; ++p) {
          double li[4], wj[4];
#pragma unroll
          for (int a = 0; a < 4; ++a) li[a] = Li[p][ty + 16 * a];
#pragma unroll
          for (int q = 0; q < 4; ++q) wj[q] = Wj[p][tx + 16 * q];
#pragma unroll
          for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[a][q] = fma(li[a], wj[q], acc[a][q]);
        }
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          const int64_t gi = i0 + ty + 16 * a;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int64_t gj = j0 + tx + 16 * q;
            if (gi < M && gj <= gi) A[gi * M + gj] -= acc[a][q];
          }
        }
        __syncthreads();
      }
    }
  }
  // inertia from the signs of D; a pivot within 1e-11 of its scale (or NaN) counts as zero
  __syncthreads();
  double pos = 0.0, neg = 0.0;
  for (int64_t i = tid; i < M; i += THREADS) {
    const double d = A[i * M + i];
    if (fabs(d) > 1e-11 * scale[i]) {
      pos += d > 0.0 ? 1.0 : 0.0;
      neg += d < 0.0 ? 1.0 : 0.0;
    }
  }
  pos = block_reduce(pos, false, red);
  neg = block_reduce(neg, false, red);
  if (tid == 0) {
    int32_t *o = inertia + 3 * (int64_t)blockIdx.x;
    o[0] = (int32_t)pos;
    o[1] = (int32_t)neg;
    o[2] = (int32_t)(M - (int64_t)pos - (int64_t)neg);
  }
}

// v := K^-1 v with the factor in the lower triangle of A (whole CTA; v in global memory, private to this CTA)
__device__ void ldl_apply_inverse(const double *A, int64_t M, double *v) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // L y = v, 32 rows at a time: rows of the block take the earlier columns (warp per row), then warp 0 solves the block
  for (int64_t I0 = 0; I0 < M; I0 += 32) {
    const int ib = (int)(M - I0 < 32 ? M - I0 : 32);
    for (int r = warp; r < ib; r += THREADS / 32) {
      const double *row = A + (I0 + r) * M;
      double s = 0.0;
      for (int64_t j = lane; j < I0; j += 32) s += row[j] * v[j];
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) v[I0 + r] -= s;
    }
    __syncthreads();
    if (warp == 0) {
      double val = lane < ib ? v[I0 + lane] : 0.0;
      for (int j = 0; j < ib; ++j) {
        const double yj = __shfl_sync(0xffffffffu, val, j);
        if (lane > j && lane < ib) val -= A[(I0 + lane) * M + I0 + j] * yj;
      }
      if (lane < ib) v[I0 + lane] = val;
    }
    __syncthreads();
  }
  for (int64_t i = tid; i < M; i += THREADS) v[i] /= A[i * M + i];
  __syncthreads();
  // L' x = y, last block first: warp 0 solves the block, then every earlier entry takes the block's columns
  for (int64_t I0 = ((M - 1) / 32) * 32; I0 >= 0; I0 -= 32) {
    const int ib = (int)(M - I0 < 32 ? M - I0 : 32);
    if (warp == 0) {
      double val = lane < ib ? v[I0 + lane] : 0.0;
      for (int j = ib - 1; j >= 0; --j) {
        const double xj = __shfl_sync(0xffffffffu, val, j);
        if (lane < j) val -= A[(I0 + j) * M + I0 + lane] * xj;
      }
      if (lane < ib) v[I0 + lane] = val;
    }
    __syncthreads();
    for (int64_t c = tid; c < I0; c += THREADS) {
      double s = 0.0;
      for (int j = 0; j < ib; ++j) s += A[(I0 + j) * M + c] * v[I0 + j];
      v[c] -= s;
    }
    __syncthreads();
  }
}

// r := b - K x with the assembled K (strict upper triangle of A + diagonal Dg); returns max_i sum_j |K_ij| when
// want_norm (every thread gets it).  tmp: M doubles of scratch.
__device__ double kkt_residual(const double *A, const double *Dg, int64_t M, const double *x, const double *b,
                               double *r, double *tmp, bool want_norm, double *red) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // column part: sum_{j<i} K_ji x_j (rows of the upper triangle, coalesced over i), and its |.| row sums
  for (int64_t i = tid; i < M; i += THREADS) {
    double s = 0.0, a = 0.0;
    for (int64_t j = 0; j < i; ++j) {
      const double kv = A[j * M + i];
      s += kv * x[j];
      a += fabs(kv);
    }
    r[i] = b[i] - Dg[i] * x[i] - s;
    tmp[i] = a + fabs(Dg[i]);
  }
  __syncthreads();
  // row part: sum_{j>i} K_ij x_j (warp per row)
  double knorm = 0.0;
  for (int64_t i = warp; i < M; i += THREADS / 32) {
    const double *row = A + i * M;
    double s = 0.0, a = 0.0;
    for (int64_t j = i + 1 + lane; j < M; j += 32) {
      s += row[j] * x[j];
      a += fabs(row[j]);
    }
    for (int o = 16; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      a += __shfl_xor_sync(0xffffffffu, a, o);
    }
    if (lane == 0) {
      r[i] -= s;
      knorm = fmax(knorm, tmp[i] + a);
    }
  }
  __syncthreads();
  if (!want_norm) return 0.0;
  return block_reduce(knorm, true, red);
}

// One CTA per selected start whose inertia is (N, M - N, 0): solve, refine once against the assembled K, check
// the normwise backward error, and form dz' W dz (dz = sol[:N]).  A start that fails gets a NaN solution.
__global__ void __launch_bounds__(THREADS) kkt_solve_kernel(const double *K, const double *Dgall, const double *Wdall,
                                                            const int32_t *starts, int64_t M, int64_t N,
                                                            const int32_t *inertia, const double *rhs, double *sol,
                                                            double *wquad, double *work) {
  __shared__ double red[THREADS / 32];
  const int c = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t b = starts[c];
  const double *A = K + b * M * M, *Dg = Dgall + b * M, *Wd = Wdall + b * N;
  const double *bv = rhs + (int64_t)c * M;
  double *out = sol + (int64_t)c * M;
  const int32_t *in = inertia + 3 * (int64_t)c;
  if (in[0] != N || in[1] != M - N || in[2] != 0) {
    for (int64_t i = tid; i < M; i += THREADS) out[i] = __longlong_as_double(0x7ff8000000000000LL);
    if (tid == 0) wquad[c] = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  double *x = work + (int64_t)c * 3 * M, *r = x + M, *tmp = r + M;
  for (int64_t i = tid; i < M; i += THREADS) x[i] = bv[i];
  __syncthreads();
  ldl_apply_inverse(A, M, x);
  kkt_residual(A, Dg, M, x, bv, r, tmp, false, red);
  ldl_apply_inverse(A, M, r);
  for (int64_t i = tid; i < M; i += THREADS) x[i] += r[i];
  __syncthreads();
  const double knorm = kkt_residual(A, Dg, M, x, bv, r, tmp, true, red);
  double rmax = 0.0, xmax = 0.0, bmax = 0.0;
  bool finite = true;
  for (int64_t i = tid; i < M; i += THREADS) {
    rmax = fmax(rmax, fabs(r[i]));
    xmax = fmax(xmax, fabs(x[i]));
    bmax = fmax(bmax, fabs(bv[i]));
    finite = finite && isfinite(x[i]);
  }
  rmax = block_reduce(rmax, true, red);
  xmax = block_reduce(xmax, true, red);
  bmax = block_reduce(bmax, true, red);
  const double nonfinite = block_reduce(finite ? 0.0 : 1.0, false, red);
  // dz' W dz = sum_i Wd_i dz_i^2 + 2 sum_{i<j<N} K_ij dz_i dz_j   (off the diagonal W and K agree)
  double q = 0.0;
  for (int64_t i = warp; i < N; i += THREADS / 32) {
    const double *row = A + i * M;
    double s = 0.0;
    for (int64_t j = i + 1 + lane; j < N; j += 32) s += row[j] * x[j];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) q += x[i] * (Wd[i] * x[i] + 2.0 * s);
  }
  q = block_reduce(q, false, red);
  const double den = knorm * xmax + bmax;
  const double eta = den > 0.0 ? rmax / den : rmax;        // b = 0: x = 0 is exact
  const bool ok = nonfinite == 0.0 && !(eta > 1e-8) && isfinite(eta);
  for (int64_t i = tid; i < M; i += THREADS) out[i] = ok ? x[i] : __longlong_as_double(0x7ff8000000000000LL);
  if (tid == 0) wquad[c] = ok ? q : __longlong_as_double(0x7ff8000000000000LL);
}

}  // namespace dnlp_kkt
