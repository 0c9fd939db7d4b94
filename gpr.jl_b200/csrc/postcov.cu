// Full posterior covariance and posterior draws (GaussianProcesses predict_f / predict_y with full_cov = true, rand):
//   Sigma_f = K** - T'T                 T = L^-1 K*, the GEMM_FWD_ROW right-hand sides of every 128-column chunk, kept
//   Sigma_y = Sigma_f + exp(2 logNoise) I
//   draws   = mu 1' + L_S Z             L_S = lower factor of make_posdef!(Sigma_f) (k_diag_factor / k_tile_gemm on a
//                                       per-call workspace, jitter ladder driven by the host like eval_pass)
#include "common.cuh"
#include "kernels.h"

namespace gprb {

// ---------------------------------------------------------------------------------------------------------
// k_post_cov: one CTA per lower 128 x 128 tile (ci >= cj) of Sigma and GP, sixteen warps with 32 x 32 register tiles.
// Prologue: the shared-memory ring holds the tile's test inputs and the accumulators start at K**(ci, cj), computed by direct
// differences in the reference's order (r2 = sum_p w_p (x_ip - x_jp)^2, like K itself - not the Gram form).
// k-loop: acc += (-T_ci)' T_cj over the nv valid rows of T on the DMMA pipe (mma.sync m8n8k4 f64 -> SASS DMMA.8x8x4); each
// KT-row chunk of T arrives as 68 x KT TMA boxes of the GEMM_FWD_ROW map (two per 128-column operand: padded pitch
// 68 = 4 mod 16, conflict-free fragment loads), ring of four stages refilled by lane 0 of warp 0 once all warps released it.
// Epilogue: Sigma = acc (+ noise on the diagonal) into the lower tile and its mirror.  Diagonal tiles compute only the ten
// warp tiles on / below the diagonal and write entries with row >= column once, mirrored: Sigma is exactly symmetric.
// Rows / columns >= m are written as the identity (the Cholesky kernels take Sigma unchanged).  The per-element summation
// order depends on nothing but the GP's own data, so a GP's Sigma does not depend on the batch it is predicted in.
// ---------------------------------------------------------------------------------------------------------
constexpr int PCV_WARPS = 16;
constexpr int PCV_THREADS = PCV_WARPS * 32;
constexpr int PCV_LDH = NB / 2 + 4;          // 68: smem pitch of one TMA box (64 test columns + 4 padding)
constexpr int PCV_HALF = KT * PCV_LDH;       // one box: KT rows of T x 68 columns
constexpr int PCV_STAGE = 4 * PCV_HALF;      // A operand (two boxes) + B operand (two boxes)
constexpr int PCV_NSTAGE = 4;
constexpr size_t PCV_SMEM = (size_t)PCV_NSTAGE * PCV_STAGE * sizeof(double) + 2 * PCV_NSTAGE * sizeof(uint64_t);
static_assert(PCV_NSTAGE * PCV_STAGE >= 2 * MAX_D * NB, "the staged test inputs of the epilogue fit the ring");

__device__ __forceinline__ void post_tile_index(int bx, int& i, int& j) {  // bx -> (i, j), j <= i, row by row
  i = (int)((__fsqrt_rn(8.0f * bx + 1.0f) - 1.0f) * 0.5f);
  while ((i + 1) * (i + 2) / 2 <= bx) ++i;
  while (i * (i + 1) / 2 > bx) --i;
  j = bx - i * (i + 1) / 2;
}

// KIND = PCV_ZERO: the leave-one-out product W = -G'G (loo.cu) - the accumulators start at zero instead of K**, no test
// inputs, theta or noise are read; T is G.
constexpr int PCV_ZERO = 4;

template <int KIND>
__global__ void __launch_bounds__(PCV_THREADS, 1) k_post_cov(const __grid_constant__ PostCovArgs g) {
  constexpr bool ZERO = KIND == PCV_ZERO;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* ring = reinterpret_cast<double*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(ring + PCV_NSTAGE * PCV_STAGE);
  uint64_t* empty = full + PCV_NSTAGE;
  __shared__ double wv[MAX_D];
  const int gl = g.g0 + blockIdx.y, gp = g.gp_off + gl, d = g.d;
  int ci, cj;
  post_tile_index(blockIdx.x, ci, cj);
  const bool diag = ci == cj;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, gq = lane >> 2, t = lane & 3;
  const int mvi = min(NB, g.m - ci * NB), mvj = min(NB, g.m - cj * NB);  // valid rows / columns of the tile
  int wm, wn;
  bool active = true;
  if (diag) {  // warp tiles on / below the diagonal only, dealt so that the four SMSPs (warp mod 4) get 3, 3, 2, 2 of them
    active = warp < 10;
    const int k = active ? warp : 0;
    wm = k < 1 ? 0 : k < 3 ? 1 : k < 6 ? 2 : 3;
    wn = k - wm * (wm + 1) / 2;
  } else {
    wm = warp >> 2;
    wn = warp & 3;
  }
  const int r0t = wm * 32, c0t = wn * 32;
  const bool masked = g.mask && g.mask[gp] != 0;  // no evaluated state: T was never computed
  double acc[4][4][2];
#pragma unroll
  for (int mi = 0; mi < 4; ++mi)
#pragma unroll
    for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
  const double* th = g.theta + (int64_t)gp * (d + 2);
  const double sf2 = ZERO ? 0.0 : exp(2.0 * th[d + 1]);
  if (!masked) {
    if (threadIdx.x == 0) {
      for (int s = 0; s < PCV_NSTAGE; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], PCV_WARPS); }
      mbar_fence_init();
    }
    if constexpr (!ZERO) {
    // prologue: the ring holds the tile's test inputs xi [d][NB] (rows) and xj [d][NB] (columns) while the accumulators
    // are set to K** by direct differences; then it becomes the operand ring of the k-loop
    const double* xi = ring;
    const double* xj = ring + MAX_D * NB;
    const double* Xs = g.Xstar + (int64_t)gl * g.xstar_stride;
    for (int idx = threadIdx.x; idx < d * NB; idx += PCV_THREADS) {
      const int p = idx / NB, s = idx - p * NB;
      ring[p * NB + s] = s < mvi ? Xs[(int64_t)(ci * NB + s) * d + p] : 0.0;
      ring[MAX_D * NB + p * NB + s] = s < mvj ? Xs[(int64_t)(cj * NB + s) * d + p] : 0.0;
    }
    if ((int)threadIdx.x < d) wv[threadIdx.x] = exp(-2.0 * th[1 + threadIdx.x]);
    __syncthreads();
    if (active) {
#pragma unroll
      for (int mi = 0; mi < 4; ++mi) {
        const int rl = r0t + mi * 8 + gq;
        if (rl >= mvi) continue;
        double r2[4][2];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) r2[ni][0] = r2[ni][1] = 0.0;
        for (int p = 0; p < d; ++p) {  // the row input is shared by the eight entries of this thread's row
          const double x = xi[p * NB + rl], w = wv[p];
#pragma unroll
          for (int ni = 0; ni < 4; ++ni) {
            const double2 y = *reinterpret_cast<const double2*>(xj + p * NB + c0t + ni * 8 + 2 * t);
            const double d0 = x - y.x, d1 = x - y.y;
            r2[ni][0] = fma(w, d0 * d0, r2[ni][0]);
            r2[ni][1] = fma(w, d1 * d1, r2[ni][1]);
          }
        }
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
          for (int e = 0; e < 2; ++e)
            if (c0t + ni * 8 + 2 * t + e < mvj) acc[mi][ni][e] = kcross<KIND>(r2[ni][e], sf2);
      }
    }
    }
    fence_proxy_async();  // the generic-proxy reads of the inputs are ordered before the TMA writes into the same ring
    __syncthreads();
    const int nch = g.nv / KT;
    const int ga = ci * g.nloc + gl, gb = cj * g.nloc + gl;
    const uint32_t bytes = (diag ? 2u : 4u) * PCV_HALF * sizeof(double);
    auto issue = [&](int c) {  // chunk c (rows c KT .. c KT + KT - 1 of T) -> stage c mod PCV_NSTAGE; lane 0 of warp 0
      double* st = ring + (c % PCV_NSTAGE) * PCV_STAGE;
      uint64_t* bar = &full[c % PCV_NSTAGE];
      mbar_expect_tx(bar, bytes);
      tma_load_3d(st, &g.tm_T68, 0, c * KT, ga, bar);
      tma_load_3d(st + PCV_HALF, &g.tm_T68, NB / 2, c * KT, ga, bar);
      if (!diag) {
        tma_load_3d(st + 2 * PCV_HALF, &g.tm_T68, 0, c * KT, gb, bar);
        tma_load_3d(st + 3 * PCV_HALF, &g.tm_T68, NB / 2, c * KT, gb, bar);
      }
    };
    if (threadIdx.x == 0)
      for (int c = 0; c < min(PCV_NSTAGE, nch); ++c) issue(c);
    // warp tiles lying entirely in the padding (rows or columns >= m) skip the DMMAs but keep the barrier protocol
    const bool compute = active && r0t < mvi && c0t < mvj;
    // row r of a 128-wide operand lives in box r >> 6 at column r & 63; a warp tile (32 rows) never straddles two boxes
    const double* abase = ring + (r0t >> 6) * PCV_HALF + (r0t & 63) + gq + t * PCV_LDH;
    const double* bbase = ring + (diag ? 0 : 2 * PCV_HALF) + (c0t >> 6) * PCV_HALF + (c0t & 63) + gq + t * PCV_LDH;
    int stage = 0;
    uint32_t phase = 0;
    for (int c = 0; c < nch; ++c) {
      mbar_wait(&full[stage], phase);
      if (compute) {
        const double* ap = abase + stage * PCV_STAGE;
        const double* bp = bbase + stage * PCV_STAGE;
#pragma unroll
        for (int k4 = 0; k4 < KT / 4; ++k4) {
          double a[4], b[4];
#pragma unroll
          for (int mi = 0; mi < 4; ++mi)  // acc = K** - T_ci' T_cj: the row operand enters negated (sign bit, integer pipe)
            a[mi] = __longlong_as_double(__double_as_longlong(ap[k4 * 4 * PCV_LDH + mi * 8]) ^ (long long)0x8000000000000000ULL);
#pragma unroll
          for (int ni = 0; ni < 4; ++ni) b[ni] = bp[k4 * 4 * PCV_LDH + ni * 8];
#pragma unroll
          for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) dmma884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[stage]);
      if (warp == 0 && c + PCV_NSTAGE < nch) {
        mbar_wait(&empty[stage], phase);
        if (lane == 0) issue(c + PCV_NSTAGE);
      }
      if (++stage == PCV_NSTAGE) { stage = 0; phase ^= 1; }
    }
  }
  const double noise = (!ZERO && g.add_noise) ? exp(2.0 * th[0]) : 0.0;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  const int64_t mpad = g.mpad;
  double* S = g.S + (int64_t)gl * mpad * mpad;
  bool nonfinite = false;
  if (active) {
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
      const int rl = r0t + mi * 8 + gq, gi = ci * NB + rl;
#pragma unroll
      for (int ni = 0; ni < 4; ++ni)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int cl = c0t + ni * 8 + 2 * t + e, gj = cj * NB + cl;
          if (diag && rl < cl) continue;  // written by its mirror
          double v;
          if (rl < mvi && cl < mvj) {
            v = masked ? qnan : acc[mi][ni][e];
            if (gi == gj) v += noise;
            nonfinite = nonfinite || !isfinite(v);
          } else {
            v = gi == gj ? 1.0 : 0.0;
          }
          S[gi + (int64_t)gj * mpad] = v;
          S[gj + (int64_t)gi * mpad] = v;
        }
    }
  }
  if (__syncthreads_or(nonfinite) && threadIdx.x == 0 && g.bad) g.bad[gl] = 1;
}

int configure_post_cov() {
  cudaError_t e = cudaFuncSetAttribute(k_post_cov<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PCV_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_post_cov<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PCV_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_post_cov<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PCV_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_post_cov<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PCV_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_post_cov<PCV_ZERO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PCV_SMEM);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_post_cov)", __FILE__, __LINE__);
  return 0;
}

int launch_loo_w(const PostCovArgs& a, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  const int Jm = a.mpad / NB;
  k_post_cov<PCV_ZERO><<<dim3(Jm * (Jm + 1) / 2, count), PCV_THREADS, PCV_SMEM, stream>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_post_cov (leave-one-out W) launch", __FILE__, __LINE__);
  return 0;
}

int launch_post_cov(const PostCovArgs& a, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  const int Jm = a.mpad / NB;
  dim3 grid(Jm * (Jm + 1) / 2, count);
  switch (a.kind) {
    case GPRB_KERNEL_SE_ARD: k_post_cov<0><<<grid, PCV_THREADS, PCV_SMEM, stream>>>(a); break;
    case GPRB_KERNEL_MAT12_ARD: k_post_cov<1><<<grid, PCV_THREADS, PCV_SMEM, stream>>>(a); break;
    case GPRB_KERNEL_MAT32_ARD: k_post_cov<2><<<grid, PCV_THREADS, PCV_SMEM, stream>>>(a); break;
    default: k_post_cov<3><<<grid, PCV_THREADS, PCV_SMEM, stream>>>(a); break;
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_post_cov launch", __FILE__, __LINE__);
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// make_posdef! on Sigma_f (one warp per listed GP): tr over the current diagonal (lane-strided partial sums, xor tree:
// every lane ends with the same value), then A_ii += 1e-6 tr / m.  The GP's failure flag is cleared for the next attempt.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_post_jitter(double* S, int32_t* fail, const int32_t* list, int m, int mpad) {
  const int g = list[blockIdx.x];
  double* A = S + (int64_t)g * mpad * mpad;
  double s = 0.0;
  for (int i = threadIdx.x; i < m; i += 32) s += A[(int64_t)i * (mpad + 1)];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  const double jit = 1e-6 * s / (double)m;
  for (int i = threadIdx.x; i < m; i += 32) A[(int64_t)i * (mpad + 1)] += jit;
  if (threadIdx.x == 0) fail[g] = 0;
}

int launch_post_jitter(double* S, int32_t* fail, const int32_t* list, int m, int mpad, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  k_post_jitter<<<count, 32, 0, stream>>>(S, fail, list, m, mpad);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_post_jitter launch", __FILE__, __LINE__);
  return 0;
}

__global__ void k_post_fail_init(int32_t* fail, const int32_t* mask, const int32_t* bad, int gp_off, int count) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < count) fail[g] = (mask[gp_off + g] != 0 || bad[g] != 0) ? -2 : 0;
}

int launch_post_fail_init(int32_t* fail, const int32_t* mask, const int32_t* bad, int gp_off, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  k_post_fail_init<<<(count + 127) / 128, 128, 0, stream>>>(fail, mask, bad, gp_off, count);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_post_fail_init launch", __FILE__, __LINE__);
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// k_post_draws: out = mu 1' + L Z, CTA = 64 test points x 64 draws of one GP, 16-deep k-slices of L and Z in shared memory,
// a thread owns 4 x 4 outputs with one accumulator each (k ascending: fixed order).  A plain FMA kernel: its m^2 ns flops
// are ns / (n^2 / m) of the T solve (1 / 400 of it at n = 2000, m = ns = 100), so it is never the limiter.
// ---------------------------------------------------------------------------------------------------------
constexpr int DR_T = 64, DR_K = 16;

__global__ void __launch_bounds__(256) k_post_draws(PostDrawArgs g) {
  __shared__ double Ls[DR_K][DR_T + 1], Zs[DR_K][DR_T + 1];
  const int gl = blockIdx.z, i0 = blockIdx.x * DR_T, s0 = blockIdx.y * DR_T;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m = g.m;
  const int64_t zoff = (int64_t)gl * g.ns * m;
  double* out = g.out + zoff;
  if (g.fail[gl] != 0) {  // no factor (no state, non-finite Sigma_f, or indefinite after 10 jitters): NaN draws
    for (int e = tid; e < DR_T * DR_T; e += 256) {
      const int i = i0 + (e & (DR_T - 1)), s = s0 + (e >> 6);
      if (i < m && s < g.ns) out[(int64_t)s * m + i] = __longlong_as_double(0x7ff8000000000000LL);
    }
    return;
  }
  const int64_t mpad = g.mpad;
  const double* L = g.L + (int64_t)gl * mpad * mpad;
  const double* Z = g.Z + zoff;
  double acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
  const int kend = min(i0 + DR_T, m);  // L(i, k) = 0 for k > i: the block's rows need k < i0 + 64 only
  for (int k0 = 0; k0 < kend; k0 += DR_K) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = tid + 256 * q;
      const int kk = e >> 6, ii = e & (DR_T - 1), k = k0 + kk;
      Ls[kk][ii] = k < m ? L[(i0 + ii) + (int64_t)k * mpad] : 0.0;  // i0 + 63 < mpad: a 64-row block never leaves the padded matrix
      const int kz = e & (DR_K - 1), ss = e >> 4, s = s0 + ss;
      Zs[kz][ss] = (k0 + kz < m && s < g.ns) ? Z[(int64_t)s * m + k0 + kz] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < DR_K; ++kk) {
      double a[4], b[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) { a[q] = Ls[kk][tx + 16 * q]; b[q] = Zs[kk][ty + 16 * q]; }
#pragma unroll
      for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[p][q] = fma(a[p], b[q], acc[p][q]);
    }
    __syncthreads();
  }
  const double* mu = g.mu + (int64_t)gl * m;
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    const int i = i0 + tx + 16 * p;
    if (i >= m) continue;
    const double mui = mu[i];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int s = s0 + ty + 16 * q;
      if (s < g.ns) out[(int64_t)s * m + i] = mui + acc[p][q];
    }
  }
}

int launch_post_draws(const PostDrawArgs& a, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  dim3 grid((a.m + DR_T - 1) / DR_T, (a.ns + DR_T - 1) / DR_T, count);
  k_post_draws<<<grid, 256, 0, stream>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_post_draws launch", __FILE__, __LINE__);
  return 0;
}

}  // namespace gprb
