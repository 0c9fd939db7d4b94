// Leave-one-out cross-validation (GaussianProcesses predict_LOO, logp_CVLOO, dlogpdθ_CVLOO), Rasmussen & Williams
// eqs. 5.10-5.13 on the K^-1 and alpha a value+gradient evaluation leaves resident.  With d = diag(K^-1):
//   mu_i  = y_i - m_i - alpha_i / d_i        var_i = 1 / d_i
//   logp  = sum_i ( 1/2 log d_i - 1/2 alpha_i^2 / d_i - 1/2 log 2pi )
//   dlogp / dtheta_j = 1/2 tr(Q' dK/dtheta_j),   Q' = u alpha' + alpha u' + 2 W
//   u = K^-1 (alpha ./ d),  c_i = -1/2 (1 + alpha_i^2 / d_i) / d_i,  W = K^-1 diag(c) K^-1 = -G'G,  G = diag(sqrt(-c)) K^-1
// The gradient is the contraction k_grad_tiles computes for Q = alpha alpha' - K^-1: it is run unchanged on a per-call
// matrix that holds K in the lower tiles and -Q' where K^-1 would be, with a zero alpha.  The stages here are the O(n)
// and O(n^2) ones around it; u is one more substitution (k_solve), W one n^3 product (k_post_cov, zero-initialised).
#include <math.h>

#include "common.cuh"
#include "kernels.h"

namespace gprb {

// ---------------------------------------------------------------------------------------------------------
// k_loo_point: one CTA per GP.  Pointwise LOO terms, v = alpha ./ d and s = sqrt(-c) (zero beyond n), and logp as a
// fixed-order sum over i < n (thread-strided partial sums, then a fixed tree): it depends on nothing but the GP's data.
// ---------------------------------------------------------------------------------------------------------
constexpr int LP_THREADS = 256;

__global__ void __launch_bounds__(LP_THREADS) k_loo_point(LooArgs g) {
  __shared__ double red[LP_THREADS];
  const int gl = blockIdx.x, gp = g.gp0 + gl;
  if (g.skip[gp] != 0) return;
  const int n = g.n, npad = g.npad;
  const double* KD = g.KinvD + (int64_t)gp * g.dinv_stride;
  const double* al = g.alpha + (int64_t)gp * npad;
  const double* y = g.ymm + (int64_t)gp * npad;
  double lp = 0.0;
  for (int i = threadIdx.x; i < npad; i += LP_THREADS) {
    double vi = 0.0, si = 0.0;
    if (i < n) {
      const int ti = i / NB, il = i - ti * NB;
      const double di = KD[(int64_t)ti * NB * NB + il + il * NB], a = al[i];
      vi = a / di;
      const double a2d = a * vi;  // alpha_i^2 / d_i
      g.mu[(int64_t)gp * n + i] = y[i] - vi;
      g.var[(int64_t)gp * n + i] = 1.0 / di;
      lp += 0.5 * log(di) - 0.5 * a2d - 0.91893853320467274;  // 1/2 log 2pi
      si = sqrt(0.5 * (1.0 + a2d) / di);
    }
    if (g.v) {
      g.v[(int64_t)gl * npad + i] = vi;
      g.s[(int64_t)gl * npad + i] = si;
    }
  }
  red[threadIdx.x] = lp;
  __syncthreads();
  for (int w = LP_THREADS / 2; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) g.logp[gp] = red[0];
}

int launch_loo_point(const LooArgs& a, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  k_loo_point<<<count, LP_THREADS, 0, stream>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_loo_point launch", __FILE__, __LINE__);
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// k_loo_expand: G(r, c) = s_r K^-1(r, c) into the right-hand-side layout of k_post_cov: block (chunk c / 128, local GP),
// row r contiguous over the 128 columns of the chunk.  CTA = 32 rows x the 128 columns of one tile column, in four 32 x 32
// steps.  Where K^-1(r, c) is stored column-contiguous (diagonal tiles, read through their symmetry, and the tiles above
// the diagonal) it is read straight; the tiles below the diagonal sit un-transposed at the mirrored tile position, so
// rows are contiguous there and the 32 x 32 block goes through shared memory.  Rows and columns >= n are written as zero.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_loo_expand(LooArgs g) {
  __shared__ double tile[32][33];
  const int gl = blockIdx.z, gp = g.gp0 + gl;
  if (g.skip[gp] != 0) return;
  const int npad = g.npad, n = g.n;
  const int r0 = blockIdx.x * 32, tj = blockIdx.y, ti = r0 / NB;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const double* A = g.A + (int64_t)gp * g.mat_stride;
  const double* s = g.s + (int64_t)gl * npad;
  double* G = g.G + ((int64_t)tj * gridDim.z + gl) * npad * PT;
  for (int q = 0; q < NB / 32; ++q) {
    const int cl0 = q * 32;  // first column of this step inside the chunk
    if (ti > tj) {
      __syncthreads();  // the previous step's reads of `tile` are done
      // K^-1(r, c) = A[(tj NB + r % NB) + (ti NB + c % NB) npad]: rows contiguous
      for (int k = ty; k < 32; k += 8)
        tile[k][tx] = A[(int64_t)(tj * NB + (r0 % NB) + tx) + (int64_t)(ti * NB + cl0 + k) * npad];
      __syncthreads();
    }
    for (int k = ty; k < 32; k += 8) {
      const int r = r0 + k, c = tj * NB + cl0 + tx;
      double val;
      if (ti > tj) val = tile[tx][k];
      else if (ti == tj) val = g.KinvD[(int64_t)gp * g.dinv_stride + (int64_t)ti * NB * NB + (c % NB) + (int64_t)(r % NB) * NB];
      else val = A[(int64_t)(ti * NB + (c % NB)) + (int64_t)(tj * NB + (r % NB)) * npad];  // K^-1(c, r), tile (tj, ti) below
      G[(int64_t)r * PT + cl0 + tx] = (r < n && c < n) ? s[r] * val : 0.0;
    }
  }
}

int launch_loo_expand(const LooArgs& a, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  k_loo_expand<<<dim3(a.npad / 32, a.J, count), 256, 0, stream>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_loo_expand launch", __FILE__, __LINE__);
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// k_loo_assemble: one CTA per 128 x 128 tile position (tr, tc) of Ap and GP.  tr >= tc: the tile of A (K) is copied.
// tr < tc: the position holds -Q' tile (tc, tr) un-transposed, -Q'(i, j) = -(u_i alpha_j + alpha_i u_j) - 2 W(i, j)
// (no contraction: the value is exactly symmetric in i and j, like W).  tr == tc also writes the full tile to KinvDp.
// Entries with a row or column >= n are zero (k_grad_tiles ignores them).
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_loo_assemble(LooArgs g) {
  const int gl = blockIdx.z, gp = g.gp0 + gl;
  if (g.skip[gp] != 0) return;
  const int tr = blockIdx.x, tc = blockIdx.y, n = g.n;
  const int64_t npad = g.npad;
  const double* A = g.A + (int64_t)gp * g.mat_stride;
  double* Ap = g.Ap + (int64_t)gl * npad * npad;
  const int rl = threadIdx.x & (NB - 1), c0 = threadIdx.x >> 7;
  if (tr >= tc) {
    for (int cl = c0; cl < NB; cl += 2) {
      const int64_t off = (int64_t)(tr * NB + rl) + (int64_t)(tc * NB + cl) * npad;
      Ap[off] = A[off];
    }
  }
  if (tr > tc) return;
  const int ti = tc, tj = tr;  // -Q' tile (ti, tj), ti >= tj
  const double* W = g.W + (int64_t)gl * npad * npad;
  const double* al = g.alpha + (int64_t)gp * npad;
  const double* u = g.u + (int64_t)gl * npad;
  const int i = ti * NB + rl;
  const double ai = i < n ? al[i] : 0.0, ui = i < n ? u[i] : 0.0;
  double* KDp = g.KinvDp + (int64_t)gl * g.dinv_stride + (int64_t)ti * NB * NB;
  for (int cl = c0; cl < NB; cl += 2) {
    const int j = tj * NB + cl;
    double q = 0.0;
    if (i < n && j < n) {
      const double sym = __dadd_rn(__dmul_rn(ui, al[j]), __dmul_rn(ai, u[j]));
      q = __dsub_rn(-sym, 2.0 * W[i + (int64_t)j * npad]);
    }
    if (ti == tj) KDp[rl + cl * NB] = q;
    else Ap[(int64_t)(tj * NB + rl) + (int64_t)(ti * NB + cl) * npad] = q;
  }
}

int launch_loo_assemble(const LooArgs& a, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  k_loo_assemble<<<dim3(a.J, a.J, count), 256, 0, stream>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_loo_assemble launch", __FILE__, __LINE__);
  return 0;
}

}  // namespace gprb
