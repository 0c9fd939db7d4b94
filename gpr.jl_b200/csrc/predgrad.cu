// Predictive gradients (gprb_predict_grad): Jacobians of the posterior mean and variance with respect to the test inputs.
// Stationary ARD kernels k = g(r2), r2 = sum_p w_p (x*_p - x_p)^2, so dk / dx*_p = 2 g'(r2) w_p (x*_p - x_p) and
//   dmu_j / dx*_p  = dm(x*_j) / dx*_p + 2 w_p sum_i alpha_i g'_ij (x*_jp - x_ip)
//   dvar_j / dx*_p = -4 w_p sum_i beta_ij g'_ij (x*_jp - x_ip),      beta = K^-1 K* = L^-T (L^-1 K*)
// The differences are formed directly: the expanded form x*_p sum_i c_i - sum_i c_i x_ip cancels catastrophically.
// beta comes from the T block of the chunk after the forward (GEMM_FWD_ROW) and backward (GEMM_BWD_ROW) DMMA chains.
#include "common.cuh"
#include "kernels.h"

namespace gprb {

constexpr int PJ_THREADS = 512;
constexpr int PJ_RT = 32;                               // training rows per staged tile
constexpr int PJ_SL = PJ_THREADS / PT;                  // 4: input-dimension slices of the accumulation phase
constexpr int PJ_PMAX = (MAX_D + PJ_SL - 1) / PJ_SL;    // input dimensions per slice (p = slice + 4 q)
constexpr int PJ_PSMALL = 8;                            // d <= 32 (CP: 26) runs the instantiation with 8 per slice
constexpr int PJ_RG = PJ_RT / PJ_SL;                    // 8: rows per thread in the pair phase

// g'(r2) = dk / d(r2).  Mat12: -s_f^2 e^-r / (2r), 0 at r = 0 (the symmetric subgradient; the pair's difference
// vector is 0 there too).
template <int KIND>
__device__ __forceinline__ double kderiv(double r2, double sf2) {
  if (KIND == GPRB_KERNEL_SE_ARD) return -0.5 * sf2 * exp_nonpos(-0.5 * r2);
  const double r = sqrt(r2);
  if (KIND == GPRB_KERNEL_MAT12_ARD) return r > 0.0 ? -0.5 * sf2 * exp_nonpos(-r) / r : 0.0;
  if (KIND == GPRB_KERNEL_MAT32_ARD) return -1.5 * sf2 * exp_nonpos(-1.7320508075688772 * r);
  const double s = 2.23606797749979 * r;
  return -(5.0 / 6.0) * sf2 * (1.0 + s) * exp_nonpos(-s);
}

// grid count, 512 threads.  Per tile of 32 training rows (its inputs, alpha and beta rows staged by one lane with bulk
// copies, double-buffered, so that the pair phase issues no global load):
//   pair phase:  thread (column j, row group) forms r2 and g' for 8 rows and stores c_a = alpha_i g', c_b = beta_ij g'
//                (c_b in place of the staged beta)
//   accumulation: thread (column j, slice s) adds c (x*_jp - x_ip) for its input dimensions p = s, s + 4, ...
// Every accumulator sees the rows in ascending order: the result does not depend on the batch.
// PMAX: input dimensions per slice the accumulators hold (registers: 3 PMAX doubles per thread).
template <int KIND, int PMAX>
__global__ void __launch_bounds__(PJ_THREADS) k_predict_jac(PredictJacArgs g) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = g.d;
  double* cb = reinterpret_cast<double*>(smem_raw);  // [2][PJ_RT][PT] beta rows of the tile, then c_b
  double* ca = cb + 2 * PJ_RT * PT;                   // [PJ_RT][PT]
  double* Xi = ca + PJ_RT * PT;                       // [2][d + 1][PJ_RT] training tiles and their alpha (row d)
  double* xsT = Xi + 2 * (d + 1) * PJ_RT;             // [d][PT] test columns
  double* wv = xsT + d * PT;                          // [MAX_D]
  uint64_t* bar = reinterpret_cast<uint64_t*>(wv + MAX_D);  // [2]
  const int gl = blockIdx.x, gp = g.gp_off + gl;
  const int j = threadIdx.x & (PT - 1), sub = threadIdx.x / PT;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (g.mask && g.mask[gp] != 0) {  // no evaluated state: NaN rows, the other GPs of the call are unaffected
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    for (int k = threadIdx.x; k < g.mc * d; k += PJ_THREADS) {
      const int64_t o = ((int64_t)gl * g.m + g.s0) * d + k;
      g.dmu[o] = qnan;
      if (g.dvar) g.dvar[o] = qnan;
    }
    return;
  }
  const double* th = g.theta + (int64_t)gp * (d + 2);
  const double* Xt = g.Xt[gp];
  const double* alpha = g.alpha + (int64_t)gp * g.npad;
  const double* beta = g.beta ? g.beta + (int64_t)gl * g.npad * PT : nullptr;
  const int ntile = (g.n + PJ_RT - 1) / PJ_RT;
  if (threadIdx.x == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); mbar_fence_init(); }
  __syncthreads();
  auto stage = [&](int t) {  // one lane, warp-uniform operands: d + 1 copies of PJ_RT doubles and the tile's beta rows
    double* dst = Xi + (t & 1) * (d + 1) * PJ_RT;
    const int64_t r0 = (int64_t)t * PJ_RT;
    mbar_expect_tx(&bar[t & 1], (uint32_t)(((d + 1) * PJ_RT + (beta ? PJ_RT * PT : 0)) * sizeof(double)));
    for (int p = 0; p < d; ++p) bulk_g2s(dst + p * PJ_RT, Xt + (int64_t)p * g.npad + r0, PJ_RT * sizeof(double), &bar[t & 1]);
    bulk_g2s(dst + d * PJ_RT, alpha + r0, PJ_RT * sizeof(double), &bar[t & 1]);
    if (beta) bulk_g2s(cb + (t & 1) * PJ_RT * PT, beta + r0 * PT, PJ_RT * PT * sizeof(double), &bar[t & 1]);
  };
  if (warp == 0 && lane == 0) stage(0);
  if (threadIdx.x < d) wv[threadIdx.x] = exp(-2.0 * th[1 + threadIdx.x]);
  const double* Xstar = g.Xstar + (int64_t)gl * g.xstar_stride + (int64_t)g.s0 * d;
  for (int idx = threadIdx.x; idx < d * PT; idx += PJ_THREADS) {
    const int p = idx / PT, s = idx - p * PT;
    xsT[idx] = s < g.mc ? Xstar[(int64_t)s * d + p] : 0.0;
  }
  __syncthreads();
  const double sf2 = exp(2.0 * th[d + 1]);
  const bool jok = j < g.mc;
  double xs[PMAX], acc_a[PMAX], acc_b[PMAX];
#pragma unroll
  for (int q = 0; q < PMAX; ++q) {
    const int p = sub + PJ_SL * q;
    xs[q] = p < d ? xsT[p * PT + j] : 0.0;
    acc_a[q] = acc_b[q] = 0.0;
  }
  for (int t = 0; t < ntile; ++t) {
    mbar_wait(&bar[t & 1], (t >> 1) & 1);
    const double* Xb = Xi + (t & 1) * (d + 1) * PJ_RT;
    double* cbt = cb + (t & 1) * PJ_RT * PT;
    // pair phase: rows sub * 8 .. sub * 8 + 7 of the tile, column j
    {
      double r2[PJ_RG];
#pragma unroll
      for (int k = 0; k < PJ_RG; ++k) r2[k] = 0.0;
      for (int p = 0; p < d; ++p) {
        const double xj = xsT[p * PT + j], wp = wv[p];
        const double2* xr = reinterpret_cast<const double2*>(Xb + p * PJ_RT + sub * PJ_RG);
#pragma unroll
        for (int k = 0; k < PJ_RG / 2; ++k) {
          const double2 v = xr[k];
          const double d0 = xj - v.x, d1 = xj - v.y;
          r2[2 * k] = fma(wp, d0 * d0, r2[2 * k]);
          r2[2 * k + 1] = fma(wp, d1 * d1, r2[2 * k + 1]);
        }
      }
#pragma unroll
      for (int k = 0; k < PJ_RG; ++k) {
        const int rl = sub * PJ_RG + k;
        const bool ok = jok && t * PJ_RT + rl < g.n;
        const double gd = kderiv<KIND>(r2[k], sf2);
        ca[rl * PT + j] = ok ? Xb[d * PJ_RT + rl] * gd : 0.0;
        cbt[rl * PT + j] = (ok && beta) ? cbt[rl * PT + j] * gd : 0.0;
      }
    }
    __syncthreads();  // c complete; every thread is done with the other Xi buffer (read in tile t - 1)
    if (t + 1 < ntile && warp == 0 && lane == 0) stage(t + 1);
    // accumulation phase
    for (int rl = 0; rl < PJ_RT; ++rl) {
      const double a = ca[rl * PT + j], b = cbt[rl * PT + j];
#pragma unroll
      for (int q = 0; q < PMAX; ++q) {
        const int p = sub + PJ_SL * q;
        if (p < d) {
          const double df = xs[q] - Xb[p * PJ_RT + rl];
          acc_a[q] = fma(a, df, acc_a[q]);
          acc_b[q] = fma(b, df, acc_b[q]);
        }
      }
    }
    __syncthreads();  // ca and this tile's buffers are rewritten by the next tiles
  }
  if (!jok) return;
  const int64_t o = ((int64_t)gl * g.m + g.s0 + j) * d;
#pragma unroll
  for (int q = 0; q < PMAX; ++q) {
    const int p = sub + PJ_SL * q;
    if (p < d) {
      g.dmu[o + p] = 2.0 * wv[p] * acc_a[q] + (g.dmstar ? g.dmstar[o + p] : 0.0);
      if (g.dvar) g.dvar[o + p] = -4.0 * wv[p] * acc_b[q];
    }
  }
}

int launch_predict_jac(const PredictJacArgs& a, int count, cudaStream_t stream) {
  if (count <= 0 || a.mc <= 0) return 0;
  const size_t smem = (3 * (size_t)PJ_RT * PT + 2 * (size_t)(a.d + 1) * PJ_RT + (size_t)a.d * PT + MAX_D) * sizeof(double) + 2 * sizeof(uint64_t);
  cudaError_t e;
#define GPRB_PJ_LAUNCH(K, P)                                                                                \
  e = cudaFuncSetAttribute(k_predict_jac<K, P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);    \
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_predict_jac)", __FILE__, __LINE__);     \
  k_predict_jac<K, P><<<count, PJ_THREADS, smem, stream>>>(a);
#define GPRB_PJ_CASE(K)                                                     \
  if (a.d <= PJ_SL * PJ_PSMALL) { GPRB_PJ_LAUNCH(K, PJ_PSMALL) }            \
  else { GPRB_PJ_LAUNCH(K, PJ_PMAX) }
  switch (a.kind) {
    case GPRB_KERNEL_SE_ARD: GPRB_PJ_CASE(0) break;
    case GPRB_KERNEL_MAT12_ARD: GPRB_PJ_CASE(1) break;
    case GPRB_KERNEL_MAT32_ARD: GPRB_PJ_CASE(2) break;
    default: GPRB_PJ_CASE(3) break;
  }
#undef GPRB_PJ_CASE
#undef GPRB_PJ_LAUNCH
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_predict_jac launch", __FILE__, __LINE__);
  return 0;
}

}  // namespace gprb
