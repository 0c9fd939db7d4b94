// K1 covariance assembly and K5 fused log-marginal-likelihood gradient (SURVEY.md section 8a rows a5, a9).
//
// Pairwise kernels over tiles of sample pairs.  The d x 128 input tiles are staged by the TMA engine (one bulk
// copy per input dimension from the dataset's transposed copy Xt[d][npad], completion on an mbarrier).
//   k_assemble_gram  (default) the cross term of r2 = |z_i|^2 + |z_j|^2 - 2 z_i.z_j on DMMA, with an exact
//                    direct-difference path for the pairs where the expansion would lose the 1e-12 parity
//   k_assemble       the all-direct-difference kernel  r2 = sum_p w_p (x_ip - x_jp)^2  (the reference's form)
//   k_grad_tiles     the gradient, always by direct differences; it never materialises Q = alpha alpha' - K^-1 or
//                    dK/dtheta:  g_noise = s_n^2 tr(Q),  g_ll_p = 1/2 w_p sum_ij Q_ij g(r_ij) (x_ip - x_jp)^2,
//                    g_lsigma = sum_ij Q_ij K_f,ij
// Per-block partial sums go to HBM and are reduced in a fixed order by a second kernel (deterministic).
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"
#include "kernels.h"

namespace gprb {

constexpr int PW_THREADS = 256;
constexpr double EPS_F64 = 2.220446049250313e-16;

template <int KIND>
__device__ __forceinline__ void kfun(double r2, double sf2, double& kf, double& gf) {
  if (KIND == GPRB_KERNEL_SE_ARD) {
    kf = sf2 * exp_nonpos(-0.5 * r2);
    gf = kf;
  } else if (KIND == GPRB_KERNEL_MAT12_ARD) {
    const double r = sqrt(r2);
    kf = sf2 * exp_nonpos(-r);
    gf = r > 0.0 ? kf / r : 0.0;
  } else if (KIND == GPRB_KERNEL_MAT32_ARD) {
    const double s = 1.7320508075688772 * sqrt(r2);
    const double e = exp_nonpos(-s);
    kf = sf2 * (1.0 + s) * e;
    gf = 3.0 * sf2 * e;
  } else {
    const double s = 2.23606797749979 * sqrt(r2);
    const double e = exp_nonpos(-s);
    kf = sf2 * (1.0 + s + 5.0 * r2 / 3.0) * e;
    gf = (5.0 / 3.0) * sf2 * (1.0 + s) * e;
  }
}

__device__ __forceinline__ void lower_tile(int bx, int& i, int& j) {
  i = (int)((__fsqrt_rn(8.0f * bx + 1.0f) - 1.0f) * 0.5f);  // approximate, corrected by the two loops below
  while ((i + 1) * (i + 2) / 2 <= bx) ++i;
  while (i * (i + 1) / 2 > bx) --i;
  j = bx - i * (i + 1) / 2;
}

// Stage Xt[:, i*128 .. +128] and Xt[:, j*128 .. +128] into smem as Xi[p][128], Xj[p][128].
__device__ __forceinline__ void stage_inputs(const double* Xt, int npad, int d, int i, int j, double* Xi, double* Xj,
                                             uint64_t* bar) {
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) mbar_expect_tx(bar, (uint32_t)(2 * d * NB * sizeof(double)));
  __syncthreads();
  const int uwarp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp-uniform operands: see k_assemble_gram
  if (uwarp < 2 && (threadIdx.x & 31) == 0) {
    double* dst = uwarp ? Xj : Xi;
    const double* src = Xt + (int64_t)(uwarp ? j : i) * NB;
    for (int q = 0; q < d; ++q) bulk_g2s(dst + q * NB, src + (int64_t)q * npad, NB * sizeof(double), bar);
  }
  mbar_wait(bar, 0);
}

// r2[a][b] for the thread's 8x8 pair block: rows {2tx,2tx+1}+32*ra, cols {2ty,2ty+1}+(CW/4)*cb of a CW-wide column block.
template <int CW>
__device__ __forceinline__ void pair_r2(const double* Xi, const double* Xj, const double* w, int d, int tx, int ty,
                                        double (&r2)[8][8]) {
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) r2[a][b] = 0.0;
  for (int p = 0; p < d; ++p) {
    double xr[8], xc[8];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const double2 v = *reinterpret_cast<const double2*>(Xi + p * NB + 32 * a + 2 * tx);
      xr[2 * a] = v.x; xr[2 * a + 1] = v.y;
      const double2 u = *reinterpret_cast<const double2*>(Xj + p * CW + (CW / 4) * a + 2 * ty);
      xc[2 * a] = u.x; xc[2 * a + 1] = u.y;
    }
    const double wp = w[p];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int b = 0; b < 8; ++b) {
        const double df = xr[a] - xc[b];
        r2[a][b] = fma(wp, df * df, r2[a][b]);
      }
  }
}

__device__ __forceinline__ int loc8(int a, int t) { return 32 * (a >> 1) + 2 * t + (a & 1); }

template <int KIND>
__global__ void __launch_bounds__(PW_THREADS, 1) k_assemble(AssembleArgs g) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* Xi = reinterpret_cast<double*>(smem_raw);
  double* Xj = Xi + g.d * NB;
  double* w = Xj + g.d * NB;
  uint64_t* bar = reinterpret_cast<uint64_t*>(w + MAX_D);
  const int gp = g.list ? g.list[blockIdx.y] : blockIdx.y;
  int ti, tj;
  lower_tile(blockIdx.x + g.tile0, ti, tj);
  const double* th = g.theta + (int64_t)gp * (g.d + 2);
  if (threadIdx.x < g.d) w[threadIdx.x] = exp(-2.0 * th[1 + threadIdx.x]);
  stage_inputs(g.Xt[gp], g.npad, g.d, ti, tj, Xi, Xj, bar);
  __syncthreads();
  const double sf2 = exp(2.0 * th[g.d + 1]);
  const double diag_add = exp(2.0 * th[0]) + EPS_F64 + g.jitter[gp];
  if (blockIdx.x == 0 && threadIdx.x == 0) {  // info -2: non-finite theta / kernel scale (also resets the flag)
    bool ok = isfinite(sf2) && isfinite(diag_add);
    for (int p = 0; p < g.d + 2; ++p) ok = ok && isfinite(th[p]);
    for (int p = 0; p < g.d; ++p) ok = ok && isfinite(w[p]);
    g.fail[gp] = ok ? 0 : -2;
  }
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double r2[8][8];
  pair_r2<NB>(Xi, Xj, w, g.d, tx, ty, r2);
  double* A = g.A + (int64_t)gp * g.mat_stride;
  const int n = g.n;
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    const int c = tj * NB + loc8(b, ty);
#pragma unroll
    for (int a = 0; a < 8; a += 2) {
      const int r = ti * NB + loc8(a, tx);
      double v[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        double kf, gf;
        kfun<KIND>(r2[a + e][b], sf2, kf, gf);
        const int rr = r + e;
        if (rr == c) kf += diag_add;
        if (rr >= n || c >= n) kf = (rr == c) ? 1.0 : 0.0;
        v[e] = kf;
      }
      *reinterpret_cast<double2*>(A + r + (int64_t)c * g.npad) = make_double2(v[0], v[1]);
      if (g.A2) *reinterpret_cast<double2*>(g.A2 + (int64_t)gp * g.mat_stride + r + (int64_t)c * g.npad) = make_double2(v[0], v[1]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Covariance assembly with the cross term on the FP64 tensor pipe (default path).
//   z_ip = sqrt(w_p) (x_ip - x_0p)         scaled inputs, centred at the dataset's first sample (constant input
//                                          dimensions become exact zeros), built in shared memory per tile
//   r2_ij = |z_i|^2 + |z_j|^2 - 2 z_i.z_j  the d-long contraction z_i.z_j runs as DMMA.8x8x4 tiles (SASS DMMA)
// The expansion loses accuracy by an absolute delta ~ (d/4 + 2) eps (|z_i|^2 + |z_j|^2) in r2.  SEArd and Matern-3/2, 5/2
// are smooth in r2, so that is a relative error of about delta / 2 in K.  Matern-1/2, k = s_f^2 exp(-r), is not: its
// relative error is delta / (2 r), and sqrt(delta) for a duplicated sample (r = 0).
// Parity with the reference's direct differences (1e-12 relative on K) is kept by a guard: pairs whose norm sum
// exceeds GRAM_SMAX and whose K is not an underflow (r2 below the per-kernel cut-off) are recomputed with direct differences of the
// raw inputs.  With trajectory data and sane length-scales that part never fires (|z|^2 << 1); extreme
// length-scales (config.json has l down to 1e-4) take the slow exact path per element.  Matern-1/2 also recomputes the
// off-diagonal pairs that are close relative to their norm sum (GRAM_CLOSE12): with delta <= 4e-15 ssum, r >= 0.02 ssum
// keeps delta / (2 r) <= 1e-13.  Consecutive states of a trajectory and repeated samples are such pairs.
// One CTA (256 threads, 8 warps of 32 x 32 register tiles) = 128 rows x 64 columns of a lower tile; two CTAs per SM.
// ---------------------------------------------------------------------------------------------------------------
constexpr int GA_THREADS = 256;
constexpr int GA_CW = 64;             // columns per CTA
constexpr int GA_LDJ = GA_CW + 4;     // padded row of the column-input tile (conflict-free B fragments)
constexpr int GA_LDC = NB + 2;        // column stride of the cross-term tile: the accumulator stores of a half-warp hit
                                      // (2 t) GA_LDC + g, distinct modulo 16 only for a stride = 2 mod 8 (132 gave 2-way conflicts)
constexpr double GRAM_SMAX = 16.0;    // (d/4 + 2) eps * 16 < 4e-14 for d <= 62
constexpr double GRAM_CLOSE12 = 4e-4; // Matern-1/2: exact path while r2 < GRAM_CLOSE12 ssum^2, i.e. r < 0.02 ssum
// Pairs whose kernel value underflows to zero are exact zeros either way and skip the exact path.  SEArd: exp(-r2/2)
// underflows beyond r2 = 1500.  Matern: k ~ exp(-c r) with c = 1, sqrt 3, sqrt 5 only underflows beyond r = 750 / c.
// The test is made on a LOWER bound of r2 (the expansion errs by <= (d/4 + 2) eps (|z_i|^2 + |z_j|^2) < 4e-15 ssum), so
// near-duplicate points far from the centre (extreme length-scales, ssum ~ 1e17) are never misclassified as far apart.
template <int KIND>
__device__ __forceinline__ double gram_r2cut() {
  return KIND == GPRB_KERNEL_SE_ARD ? 1500.0 : KIND == GPRB_KERNEL_MAT12_ARD ? 562500.0 : KIND == GPRB_KERNEL_MAT32_ARD ? 187500.0 : 112500.0;
}

// CTAS = resident CTAs per SM the kernel is compiled for: 3 (80 registers, a few spilled words in the prologue) whenever
// three CTAs' shared memory fits an SM (d <= 44, up to 72 KB each:5.7 -> 5.15 ms per 400 GPs at d = 26, the phases of
// three CTAs interleave better than those of two), else 2.
template <int KIND, int CTAS>
__global__ void __launch_bounds__(GA_THREADS, CTAS) k_assemble_gram(AssembleArgs g) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = g.d, dpad = (d + 3) & ~3;
  double* Zi = reinterpret_cast<double*>(smem_raw);   // [dpad][LDS_T]  row-input tile, one padded row per dimension
  double* Zj = Zi + dpad * LDS_T;                      // [dpad][GA_LDJ] column-input tile
  const int zreg = max(dpad * (LDS_T + GA_LDJ), GA_CW * GA_LDC);  // the input tiles' space later holds the cross-term tile
  double* w = Zi + zreg;                               // [MAX_D + 2]  w_p
  double* sw = w + MAX_D + 2;                          // [MAX_D + 2]  sqrt(w_p)
  double* x0 = sw + MAX_D + 2;                         // [MAX_D + 2]  centre: first sample of the dataset
  double* ni = x0 + MAX_D + 2;                         // [NB]     |z_i|^2
  double* nj = ni + NB;                                // [GA_CW]  |z_j|^2
  uint64_t* bar = reinterpret_cast<uint64_t*>(nj + GA_CW);
  const int gp = g.list ? g.list[blockIdx.y] : blockIdx.y;
  const int tile = (blockIdx.x >> 1) + g.tile0, half = blockIdx.x & 1;
  int ti, tj;
  lower_tile(tile, ti, tj);
  const double* th = g.theta + (int64_t)gp * (d + 2);
  const double* Xt = g.Xt[gp];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c0 = tj * NB + half * GA_CW;  // first global column of this CTA
  if (tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
  __syncthreads();
  if (tid == 0) mbar_expect_tx(bar, (uint32_t)(d * (NB + GA_CW) * sizeof(double)));
  __syncthreads();
  {  // lane 0 of warps 0-3 issues the copies with warp-uniform operands (per-lane addresses would serialise the
     // uniform-datapath UBLKCP through an ELECT / R2UR.BROADCAST loop over the lanes): warps 0, 1 the row tile, 2, 3 the column tile
    const int uwarp = __shfl_sync(0xffffffffu, warp, 0);
    if (uwarp < 4 && lane == 0) {
      const int half_d = (d + 1) >> 1, k0 = (uwarp & 1) * half_d, k1 = (uwarp & 1) ? d : half_d;
      if (uwarp < 2) for (int k = k0; k < k1; ++k) bulk_g2s(Zi + k * LDS_T, Xt + (int64_t)k * g.npad + (int64_t)ti * NB, NB * sizeof(double), bar);
      else for (int k = k0; k < k1; ++k) bulk_g2s(Zj + k * GA_LDJ, Xt + (int64_t)k * g.npad + c0, GA_CW * sizeof(double), bar);
    }
  }
  if (tid < d) {
    const double wp = exp(-2.0 * th[1 + tid]);  // SEArd stores il2 = exp(-2 ll)
    w[tid] = wp;
    sw[tid] = sqrt(wp);
    x0[tid] = Xt[(int64_t)tid * g.npad];
  }
  for (int k = d * LDS_T + tid; k < dpad * LDS_T; k += GA_THREADS) Zi[k] = 0.0;  // zero rows d .. dpad-1
  for (int k = d * GA_LDJ + tid; k < dpad * GA_LDJ; k += GA_THREADS) Zj[k] = 0.0;
  const double sf2 = exp(2.0 * th[d + 1]);
  const double diag_add = exp(2.0 * th[0]) + EPS_F64 + g.jitter[gp];
  mbar_wait(bar, 0);
  __syncthreads();
  if (blockIdx.x == 0 && tid == 0) {  // info -2: non-finite theta / kernel scale (also resets the flag)
    bool ok = isfinite(sf2) && isfinite(diag_add);
    for (int p = 0; p < d + 2; ++p) ok = ok && isfinite(th[p]);
    for (int p = 0; p < d; ++p) ok = ok && isfinite(w[p]);
    g.fail[gp] = ok ? 0 : -2;
  }
  // scale + centre in place, then the squared norms (thread r: row r, threads < 64: column r as well)
  for (int k = tid; k < d * NB; k += GA_THREADS) {
    const int p = k >> 7, r = k & (NB - 1);
    Zi[p * LDS_T + r] = sw[p] * (Zi[p * LDS_T + r] - x0[p]);
  }
  for (int k = tid; k < d * GA_CW; k += GA_THREADS) {
    const int p = k >> 6, r = k & (GA_CW - 1);
    Zj[p * GA_LDJ + r] = sw[p] * (Zj[p * GA_LDJ + r] - x0[p]);
  }
  __syncthreads();
  if (tid < NB) {
    double s = 0.0;
    for (int p = 0; p < d; ++p) { const double z = Zi[p * LDS_T + tid]; s = fma(z, z, s); }
    ni[tid] = s;
  } else if (tid < NB + GA_CW) {
    double q = 0.0;
    for (int p = 0; p < d; ++p) { const double z = Zj[p * GA_LDJ + tid - NB]; q = fma(z, z, q); }
    nj[tid - NB] = q;
  }
  // cross term z_i . z_j on the tensor pipe
  const int wm = warp & 3, wn = warp >> 2;
  const int gq = lane >> 2, t = lane & 3;
  double acc[4][4][2];
#pragma unroll
  for (int mi = 0; mi < 4; ++mi)
#pragma unroll
    for (int ni_ = 0; ni_ < 4; ++ni_) acc[mi][ni_][0] = acc[mi][ni_][1] = 0.0;
  for (int k4 = 0; k4 < dpad / 4; ++k4) {
    double a[4], b[4];
    const double* ap = Zi + (k4 * 4 + t) * LDS_T + wm * 32 + gq;
    const double* bp = Zj + (k4 * 4 + t) * GA_LDJ + wn * 32 + gq;
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) a[mi] = ap[mi * 8];
#pragma unroll
    for (int ni_ = 0; ni_ < 4; ++ni_) b[ni_] = bp[ni_ * 8];
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
      for (int ni_ = 0; ni_ < 4; ++ni_) dmma884(acc[mi][ni_][0], acc[mi][ni_][1], a[mi], b[ni_]);
  }
  __syncthreads();  // norms visible; every warp is done with the input tiles: their space becomes the cross-term tile
  double* Cs = Zi;  // [GA_CW][GA_LDC] column-major z_i.z_j
#pragma unroll
  for (int mi = 0; mi < 4; ++mi)
#pragma unroll
    for (int ni_ = 0; ni_ < 4; ++ni_) {
      const int rl = wm * 32 + mi * 8 + gq, cl = wn * 32 + ni_ * 8 + 2 * t;
      Cs[cl * GA_LDC + rl] = acc[mi][ni_][0];
      Cs[(cl + 1) * GA_LDC + rl] = acc[mi][ni_][1];
    }
  __syncthreads();
  // epilogue, rolled (a fully unrolled register epilogue is instruction-fetch bound): thread = (row, 32-column half);
  // consecutive lanes write consecutive rows of one column (full 128 B lines)
  double* A = g.A + (int64_t)gp * g.mat_stride;
  const int n = g.n;
  const int rl = tid & (NB - 1), rr = ti * NB + rl, cbeg = (tid >> 7) * (GA_CW / 2);
  const double nr = ni[rl];
#pragma unroll 8
  for (int cl = cbeg; cl < cbeg + GA_CW / 2; ++cl) {
    const int c = c0 + cl;
    const double ssum = nr + nj[cl];
    double r2 = fmax(ssum - 2.0 * Cs[cl * GA_LDC + rl], 0.0);
    // r2 - 4e-15 ssum is a lower bound of the true r2: a pair is never misclassified as far apart
    const bool far_out = ssum > GRAM_SMAX;
    const bool close12 = KIND == GPRB_KERNEL_MAT12_ARD && rr != c && r2 - 4e-15 * ssum < GRAM_CLOSE12 * ssum * ssum;
    if ((far_out || close12) && r2 - 4e-15 * ssum < gram_r2cut<KIND>() && rr < n && c < n) {  // exact path: direct differences of the raw inputs
      r2 = 0.0;
      for (int p = 0; p < d; ++p) {
        const double df = Xt[(int64_t)p * g.npad + rr] - Xt[(int64_t)p * g.npad + c];
        r2 = fma(w[p], df * df, r2);
      }
    }
    double kf, gf;
    kfun<KIND>(r2, sf2, kf, gf);
    if (rr == c) kf = sf2 + diag_add;            // r2 is exactly zero on the diagonal
    if (rr >= n || c >= n) kf = (rr == c) ? 1.0 : 0.0;
    A[rr + (int64_t)c * g.npad] = kf;
    if (g.A2) g.A2[(int64_t)gp * g.mat_stride + rr + (int64_t)c * g.npad] = kf;
  }
}

// Gradient tiles.  One CTA (128 threads) = 128 rows x 32 columns of one lower tile; two CTAs per SM.
// The K^-1 block, the K block and both input tiles are landed in shared memory by bulk async copies (TMA engine,
// 1 KB per column), so all 98 KB of a block are in flight at once and the HBM latency of one CTA hides behind the
// FP64 phase (3 d flops per pair) of the other.  (Register-destination loads cannot do this: with the 8x4 pair
// block in registers the compiler keeps only a handful of loads in flight and the kernel becomes latency bound.)
// Thread = 8 x 4 pairs: rows {2tx,2tx+1} + 32a (a < 4), columns {2ty,2ty+1} + 16cb (cb < 2).
constexpr int GRAD_CW = NB / GRAD_PARTS_PER_TILE;  // 32
constexpr int GRAD_THREADS = 128;
static_assert(GRAD_CW == 32, "thread mapping below assumes 32-column blocks");

constexpr int GRAD_DH = 32;  // input dimensions resident at a time: d > 32 (FB: d = 52) streams its input tiles in two passes
                             // so that the CTA stays at ~105 KB of smem and two CTAs fit an SM for every d

// LEAN (every d but 31 and 32: the rows of one pass, <= 32, fit the K^-1 landing zone that the reduction reuses): the K block is not landed in
// shared memory but prefetched into 32 registers per thread before the wait on the bulk copies - 66 KB per CTA, so THREE
// CTAs share an SM and the FP64 phase of one always has the copies / reductions of two others to hide behind (with two
// CTAs per SM the DFMA pipe sat at 56 %: a CTA spends longer outside its FP64 phase than inside).
template <int KIND, bool MULTI, bool LEAN>  // MULTI = false: d <= GRAD_DH, one resident pass (the common case compiles without the pass logic)
__global__ void __launch_bounds__(GRAD_THREADS, LEAN ? 3 : 2) k_grad_tiles(GradArgs g) {
  constexpr int CW = GRAD_CW, NT = GRAD_THREADS, NQ = NB / CW, DH = MULTI ? GRAD_DH : MAX_D + 2;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = g.d, dh = min(d, DH), npass = MULTI ? (d + DH - 1) / DH : 1;
  double* Ki = reinterpret_cast<double*>(smem_raw);  // [CW][NB] K^-1 block, column-major; reused as `red` afterwards
  double* Kb = Ki + CW * NB;                          // [CW][NB] K block (SEArd only; absent in the lean layout)
  double* Xi = LEAN ? Kb : Kb + CW * NB;              // [dh][NB]  input tile of the current pass
  double* Xj = Xi + dh * NB;                          // [dh][CW]
  double* w = Xj + dh * CW;                           // [MAX_D]
  uint64_t* bar = reinterpret_cast<uint64_t*>(w + MAX_D);
  double* red = Ki;                                   // [rows of one pass (+ 2)][NT]: <= 32 rows in the lean layout, <= 34 otherwise
  const int gp = g.list ? g.list[blockIdx.y] : blockIdx.y;
  if (g.fail[gp] != 0) return;  // failed factorisation: k_grad_reduce reports NaN, nothing to sum
  const int tile = blockIdx.x / NQ, cq = blockIdx.x - tile * NQ;
  int ti, tj;
  lower_tile(tile, ti, tj);
  constexpr bool REUSE_K = (KIND == GPRB_KERNEL_SE_ARD);
  const double* th = g.theta + (int64_t)gp * (d + 2);
  const double* Xt = g.Xt[gp];
  const int cbase = cq * CW;  // first column of this block inside the tile
  const double* Kt = g.A + (int64_t)gp * g.mat_stride + (int64_t)ti * NB + (int64_t)(tj * NB + cbase) * g.npad;  // K block
  const double* Kinv;  // K^-1 block: tile (ti,tj), ti > tj, lives un-transposed at tile position (tj,ti); diagonal tiles in KinvD
  int64_t ldk;
  if (ti == tj) { ldk = NB; Kinv = g.KinvD + (int64_t)gp * g.dinv_stride + (int64_t)ti * NB * NB + (int64_t)cbase * ldk; }
  else { ldk = g.npad; Kinv = g.A + (int64_t)gp * g.mat_stride + (int64_t)tj * NB + ((int64_t)ti * NB + cbase) * ldk; }
  if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_fence_init(); }
  __syncthreads();
  const int uwarp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp index, provably warp-uniform
  const bool lane0 = (threadIdx.x & 31) == 0;
  // Input tiles of pass q (dimensions q*DH ..): one bulk copy per dimension and tile.  `cur` = resident pass.
  uint32_t parity = 0;
  int cur = 0;
  auto issue_x = [&](int q, uint32_t extra_bytes) {
    const int p0 = q * DH, pc = min(DH, d - p0);
    if (threadIdx.x == 0) mbar_expect_tx(bar, (uint32_t)(pc * (NB + CW) * sizeof(double)) + extra_bytes);
    __syncthreads();
    // Copies are issued by lane 0 of a warp with warp-uniform operands (uwarp): with per-lane addresses the compiler
    // serialises the uniform-datapath UBLKCP through an ELECT / R2UR.BROADCAST loop over the lanes (~90 cycles per copy).
    if (uwarp == 2 && lane0) {
      const double* src = Xt + (int64_t)p0 * g.npad + (int64_t)ti * NB;
      for (int k = 0; k < pc; ++k) bulk_g2s(Xi + k * NB, src + (int64_t)k * g.npad, NB * sizeof(double), bar);
    } else if (uwarp == 3 && lane0) {
      const double* src = Xt + (int64_t)p0 * g.npad + (int64_t)tj * NB + cbase;
      for (int k = 0; k < pc; ++k) bulk_g2s(Xj + k * CW, src + (int64_t)k * g.npad, CW * sizeof(double), bar);
    }
  };
  auto need_pass = [&](int q) {  // make pass q resident (no-op when it already is)
    if (!MULTI || q == cur) return;
    __syncthreads();  // everyone is done reading the resident tiles
    issue_x(q, 0);
    mbar_wait(bar, parity);
    parity ^= 1;
    cur = q;
  };
  // first batch: 32 + 32 matrix columns and the input tiles of pass 0, all in flight at once
  constexpr bool LAND_K = REUSE_K && !LEAN;
  issue_x(0, (uint32_t)((LAND_K ? 2 : 1) * CW * NB * sizeof(double)));
  if (LAND_K) {  // warp 0: K^-1 block, warp 1: K block
    if (uwarp == 0 && lane0) {
#pragma unroll 4
      for (int k = 0; k < CW; ++k) bulk_g2s(Ki + k * NB, Kinv + (int64_t)k * ldk, NB * sizeof(double), bar);
    } else if (uwarp == 1 && lane0) {
#pragma unroll 4
      for (int k = 0; k < CW; ++k) bulk_g2s(Kb + k * NB, Kt + (int64_t)k * g.npad, NB * sizeof(double), bar);
    }
  } else if (uwarp < 2 && lane0) {  // warps 0 and 1: one half of the K^-1 block each
    const int k0 = uwarp * (CW / 2);
#pragma unroll 4
    for (int k = k0; k < k0 + CW / 2; ++k) bulk_g2s(Ki + k * NB, Kinv + (int64_t)k * ldk, NB * sizeof(double), bar);
  }
  if (threadIdx.x < d) w[threadIdx.x] = exp(-2.0 * th[1 + threadIdx.x]);
  const double sf2 = exp(2.0 * th[d + 1]);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double2 kreg[4][4];  // lean layout: this thread's 8 x 4 entries of the K block, in flight while the bulk copies land
  if (LEAN && REUSE_K) {
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
      for (int a2 = 0; a2 < 4; ++a2)
        kreg[b][a2] = *reinterpret_cast<const double2*>(Kt + (int64_t)(16 * (b >> 1) + 2 * ty + (b & 1)) * g.npad + loc8(2 * a2, tx));
  }
  const double* alpha = g.alpha + (int64_t)gp * g.npad;
  const int n = g.n;
  double ar[8], ac[4];
#pragma unroll
  for (int a = 0; a < 8; ++a) ar[a] = alpha[ti * NB + loc8(a, tx)];
#pragma unroll
  for (int b = 0; b < 4; ++b) ac[b] = alpha[tj * NB + cbase + 16 * (b >> 1) + 2 * ty + (b & 1)];
  mbar_wait(bar, parity);
  parity ^= 1;
  __syncthreads();  // w visible
  double m[8][4];
  if (!REUSE_K) {  // Matern needs r itself: distances from the staged inputs (m holds r2 for now)
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) m[a][b] = 0.0;
    for (int q = 0; q < npass; ++q) {
      need_pass(q);
      const int p0 = q * DH, pc = min(DH, d - p0);
      for (int p = 0; p < pc; ++p) {
        double xr[8], xc[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          const double2 v = *reinterpret_cast<const double2*>(Xi + p * NB + 32 * a + 2 * tx);
          xr[2 * a] = v.x; xr[2 * a + 1] = v.y;
        }
#pragma unroll
        for (int cb = 0; cb < 2; ++cb) {
          const double2 u = *reinterpret_cast<const double2*>(Xj + p * CW + 16 * cb + 2 * ty);
          xc[2 * cb] = u.x; xc[2 * cb + 1] = u.y;
        }
        const double wp = w[p0 + p];
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            const double df = xr[a] - xc[b];
            m[a][b] = fma(wp, df * df, m[a][b]);
          }
      }
    }
  }
  // phase 1: m_ij = (alpha_i alpha_j - Kinv_ij) g(r_ij).  SEArd: dK/dll_p = K_f w_p Delta_p^2 and K_f,ij (i != j) is
  // still resident in the lower tiles of A, so the distance pass and the exp are skipped.
  double s_sig = 0.0, s_tr = 0.0;
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    const int cl = 16 * (b >> 1) + 2 * ty + (b & 1), c = tj * NB + cbase + cl;
#pragma unroll
    for (int a = 0; a < 8; a += 2) {
      const int rl = loc8(a, tx), r = ti * NB + rl;
      const double2 kv = *reinterpret_cast<const double2*>(Ki + cl * NB + rl);
      const double kin[2] = {kv.x, kv.y};
      double kst[2] = {0.0, 0.0};
      if (REUSE_K) {
        const double2 ks = LEAN ? kreg[b][a >> 1] : *reinterpret_cast<const double2*>(Kb + cl * NB + rl);
        kst[0] = ks.x; kst[1] = ks.y;
      }
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int rr = r + e;
        double kf, gf;
        if (REUSE_K) { kf = (rr == c) ? sf2 : kst[e]; gf = kf; }
        else kfun<KIND>(m[a + e][b], sf2, kf, gf);
        double q = ar[a + e] * ac[b] - kin[e];
        if (rr >= n || c >= n) { q = 0.0; kf = 0.0; gf = 0.0; }
        s_sig = fma(q, kf, s_sig);
        if (rr == c) s_tr += q;
        m[a + e][b] = q * gf;
      }
    }
  }
  __syncthreads();  // every thread is done with the landed blocks: the space becomes `red`
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const double wt = (ti == tj) ? 1.0 : 2.0;
  double* part = g.part + ((int64_t)gp * gridDim.x + blockIdx.x) * (d + 2);
  // phase 2 (FP64 pipe): per-dimension weighted sums; one scalar per (p, thread) parked in smem.  Passes start with
  // the resident one (the last pass after a Matern distance sweep, pass 0 otherwise).
  for (int qq = 0; qq < npass; ++qq) {
    const int q = (cur + qq) % npass;
    need_pass(q);
    const int p0 = q * DH, pc = min(DH, d - p0);
    for (int p = 0; p < pc; ++p) {
      double xr[8], xc[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const double2 v = *reinterpret_cast<const double2*>(Xi + p * NB + 32 * a + 2 * tx);
        xr[2 * a] = v.x; xr[2 * a + 1] = v.y;
      }
#pragma unroll
      for (int cb = 0; cb < 2; ++cb) {
        const double2 u = *reinterpret_cast<const double2*>(Xj + p * CW + 16 * cb + 2 * ty);
        xc[2 * cb] = u.x; xc[2 * cb + 1] = u.y;
      }
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;  // four independent FMA chains (two left the DFMA latency exposed)
#pragma unroll
      for (int a = 0; a < 8; a += 2)
#pragma unroll
        for (int b = 0; b < 4; b += 2) {
          const double d0 = xr[a] - xc[b], d1 = xr[a + 1] - xc[b];
          const double d2 = xr[a] - xc[b + 1], d3 = xr[a + 1] - xc[b + 1];
          s0 = fma(m[a][b], d0 * d0, s0);
          s1 = fma(m[a + 1][b], d1 * d1, s1);
          s2 = fma(m[a][b + 1], d2 * d2, s2);
          s3 = fma(m[a + 1][b + 1], d3 * d3, s3);
        }
      red[p * NT + threadIdx.x] = (s0 + s1) + (s2 + s3);
    }
    // Every pass is reduced on its own (its rows never exceed the 32 the lean landing zone holds); the two scalar sums
    // ride with the last - shortest - pass.  The __syncthreads at the top of need_pass orders the next pass's writes.
    int nrows = pc;
    if (q == npass - 1) {
      red[pc * NT + threadIdx.x] = s_sig;
      red[(pc + 1) * NT + threadIdx.x] = s_tr;
      nrows += 2;
    }
    __syncthreads();
    // fixed-order block reduction: warp v sums rows v, v + 4, ...
    for (int row = warp; row < nrows; row += NT / 32) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < NT / 32; ++k) s += red[row * NT + lane + 32 * k];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
      if (lane == 0) {
        // part layout: [0] trace(Q) part, [1..d] sum Q g Delta_p^2, [d+1] sum Q K_f
        if (row < pc) part[1 + p0 + row] = wt * s;
        else if (row == pc) part[d + 1] = wt * s;
        else part[0] = s;  // trace lives on diagonal tiles only (weight 1)
      }
    }
  }
}

__global__ void k_grad_reduce(GradArgs g) {
  const int gp = g.list ? g.list[blockIdx.x] : blockIdx.x;
  const int d = g.d, P = d + 2;
  const int ntiles = g.J * (g.J + 1) / 2 * (NB / GRAD_CW);  // partial blocks written by k_grad_tiles
  const double* th = g.theta + (int64_t)gp * P;
  const double* part = g.part + (int64_t)gp * ntiles * P;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    double s = 0.0;
    for (int t = 0; t < ntiles; ++t) s += part[(int64_t)t * P + p];
    double v;
    if (p == 0) v = exp(2.0 * th[0]) * s;                 // dmll_noise: exp(2 logNoise) tr(Q), no eps
    else if (p <= d) v = 0.5 * exp(-2.0 * th[p]) * s;      // 1/2 w_p sum Q g Delta_p^2
    else v = s;                                            // dK/dlsigma = 2 K_f
    if (g.fail[gp] != 0) v = __longlong_as_double(0x7ff8000000000000LL);
    g.grad[(int64_t)gp * P + p] = v;
  }
}

__global__ void k_transpose_inputs(const double* X, double* Xt, int n, int npad, int d) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)npad * d) return;
  const int p = (int)(idx / npad), r = (int)(idx % npad);
  Xt[idx] = r < n ? X[(int64_t)r * d + p] : 0.0;
}

// all datasets of a slab in one launch: blockIdx.y = dataset
__global__ void k_transpose_inputs_batched(const double* X, double* Xt, int n, int npad, int d) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)npad * d) return;
  const int p = (int)(idx / npad), r = (int)(idx % npad);
  X += (int64_t)blockIdx.y * n * d;
  Xt += (int64_t)blockIdx.y * npad * d;
  Xt[idx] = r < n ? X[(int64_t)r * d + p] : 0.0;
}

// make_posdef!: K_ii += 1e-6 tr(K)/n, cumulative.  For a stationary kernel tr(K)/n = s_f^2 + (s_n^2 + eps + jitter)
// exactly, so the increment needs no pass over the matrix; the next assembly applies it.
__global__ void k_add_jitter(const double* theta, double* jitter, const int32_t* list, int d, int count) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  const int gp = list[k];
  const double* th = theta + (int64_t)gp * (d + 2);
  const double mean_diag = exp(2.0 * th[d + 1]) + exp(2.0 * th[0]) + EPS_F64 + jitter[gp];
  jitter[gp] += 1e-6 * mean_diag;
}

static size_t pw_smem(int d, bool grad, bool lean = false) {
  size_t doubles = grad ? (size_t)(lean ? 1 : 2) * GRAD_CW * NB + (size_t)std::min(d, GRAD_DH) * (NB + GRAD_CW) + MAX_D : (size_t)2 * d * NB + MAX_D;
  return doubles * sizeof(double) + 16;
}

template <typename K>
static int set_smem(K kernel, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute", __FILE__, __LINE__);
  return 0;
}

int launch_assemble(const AssembleArgs& a, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  // GPRB200_ASSEMBLY=direct selects the all-direct-difference kernel (A/B comparisons, tests); default is the DMMA path
  static const bool direct = [] { const char* e = getenv("GPRB200_ASSEMBLY"); return e && e[0] == 'd'; }();
  int rc = 0;
  if (!direct) {
    const int dpad = (a.d + 3) & ~3;
    const size_t zreg = std::max((size_t)dpad * (LDS_T + GA_LDJ), (size_t)GA_CW * GA_LDC);  // input tiles, later the cross-term tile
    const size_t smem = (zreg + 3 * (MAX_D + 2) + NB + GA_CW) * sizeof(double) + 16;
    dim3 grid((a.J * (a.J + 1) / 2 - a.tile0) * (NB / GA_CW), count);
    const bool three = 3 * (smem + 1024) <= 227 * 1024;  // three CTAs per SM fit (1 KB per CTA is reserved by the driver)
#define GPRB_GA_CASE(K)                                                                  \
  if (three) {                                                                           \
    rc = set_smem(k_assemble_gram<K, 3>, smem);                                          \
    if (!rc) k_assemble_gram<K, 3><<<grid, GA_THREADS, smem, stream>>>(a);               \
  } else {                                                                               \
    rc = set_smem(k_assemble_gram<K, 2>, smem);                                          \
    if (!rc) k_assemble_gram<K, 2><<<grid, GA_THREADS, smem, stream>>>(a);               \
  }
    switch (a.kind) {
      case GPRB_KERNEL_SE_ARD: GPRB_GA_CASE(0) break;
      case GPRB_KERNEL_MAT12_ARD: GPRB_GA_CASE(1) break;
      case GPRB_KERNEL_MAT32_ARD: GPRB_GA_CASE(2) break;
      default: GPRB_GA_CASE(3) break;
    }
#undef GPRB_GA_CASE
  } else {
    const size_t smem = pw_smem(a.d, false);
    dim3 grid(a.J * (a.J + 1) / 2 - a.tile0, count);
    switch (a.kind) {
      case GPRB_KERNEL_SE_ARD: rc = set_smem(k_assemble<0>, smem); if (!rc) k_assemble<0><<<grid, PW_THREADS, smem, stream>>>(a); break;
      case GPRB_KERNEL_MAT12_ARD: rc = set_smem(k_assemble<1>, smem); if (!rc) k_assemble<1><<<grid, PW_THREADS, smem, stream>>>(a); break;
      case GPRB_KERNEL_MAT32_ARD: rc = set_smem(k_assemble<2>, smem); if (!rc) k_assemble<2><<<grid, PW_THREADS, smem, stream>>>(a); break;
      default: rc = set_smem(k_assemble<3>, smem); if (!rc) k_assemble<3><<<grid, PW_THREADS, smem, stream>>>(a); break;
    }
  }
  if (rc) return rc;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_assemble launch", __FILE__, __LINE__);
  return 0;
}

int launch_grad(const GradArgs& a, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  // lean layout (three CTAs per SM) whenever the (d + 2) x 128 reduction buffer fits the K^-1 landing zone;
  // GPRB200_GRAD_LEAN=0 forces the two-block layout (A/B comparisons)
  static const bool allow_lean = [] { const char* e = getenv("GPRB200_GRAD_LEAN"); return !(e && e[0] == '0'); }();
  const bool lean = allow_lean && (a.d + 2 <= GRAD_CW || a.d > GRAD_DH);  // single pass of <= 30 dims, or passes of 32 + a short last one
  const size_t smem = pw_smem(a.d, true, lean);
  dim3 grid(a.J * (a.J + 1) / 2 * (NB / GRAD_CW), count);
  int rc = 0;
#define GPRB_GRAD_LAUNCH(K, M, L)                                         \
  rc = set_smem(k_grad_tiles<K, M, L>, smem);                             \
  if (!rc) k_grad_tiles<K, M, L><<<grid, GRAD_THREADS, smem, stream>>>(a);
#define GPRB_GRAD_CASE(K)                                                 \
  if (a.d <= GRAD_DH) {                                                   \
    if (lean) { GPRB_GRAD_LAUNCH(K, false, true) }                        \
    else { GPRB_GRAD_LAUNCH(K, false, false) }                            \
  } else if (lean) { GPRB_GRAD_LAUNCH(K, true, true) }                    \
  else { GPRB_GRAD_LAUNCH(K, true, false) }
  switch (a.kind) {
    case GPRB_KERNEL_SE_ARD: GPRB_GRAD_CASE(0) break;
    case GPRB_KERNEL_MAT12_ARD: GPRB_GRAD_CASE(1) break;
    case GPRB_KERNEL_MAT32_ARD: GPRB_GRAD_CASE(2) break;
    default: GPRB_GRAD_CASE(3) break;
  }
#undef GPRB_GRAD_CASE
#undef GPRB_GRAD_LAUNCH
  if (rc) return rc;
  k_grad_reduce<<<count, 64, 0, stream>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_grad launch", __FILE__, __LINE__);
  return 0;
}

int launch_transpose_inputs(const double* X, double* Xt, int n, int npad, int d, cudaStream_t stream) {
  const int64_t total = (int64_t)npad * d;
  k_transpose_inputs<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(X, Xt, n, npad, d);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_transpose_inputs launch", __FILE__, __LINE__);
  return 0;
}

int launch_transpose_inputs_batched(const double* X, double* Xt, int n, int npad, int d, int count, cudaStream_t stream) {
  const int64_t total = (int64_t)npad * d;
  dim3 grid((unsigned)((total + 255) / 256), count);
  k_transpose_inputs_batched<<<grid, 256, 0, stream>>>(X, Xt, n, npad, d);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_transpose_inputs_batched launch", __FILE__, __LINE__);
  return 0;
}

int launch_add_jitter(const double* theta, double* jitter, const int32_t* list, int d, int count, cudaStream_t stream) {
  if (count <= 0) return 0;
  k_add_jitter<<<(count + 127) / 128, 128, 0, stream>>>(theta, jitter, list, d, count);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_add_jitter launch", __FILE__, __LINE__);
  return 0;
}

}  // namespace gprb
