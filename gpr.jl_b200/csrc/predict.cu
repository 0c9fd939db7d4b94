// K6 posterior prediction (SURVEY.md section 8a row a11; reference call examples/utils/predictdynamics.jl:13):
//   k*_r = k(X[:,r], x*) ;  mu* = m(x*) + k*' alpha ;  var* = max(s_f^2 - |L^-1 k*|^2, 0) + exp(2 logNoise)
// Two paths:
//   k_predict        (m <= 8 with the triangular inverse V resident): one CTA handles PS test columns of one GP,
//                    cross-covariances in shared memory, fused mean dot, variance streams V once (GEMV-like, HBM bound)
//   k_predict_cross + GEMM_FWD_ROW tiles + k_predict_finish   (everything else): chunks of 128 test columns, the
//                    variance is the blocked forward substitution L^-1 K* on the DMMA pipe (FP64 bound, n^2 flop/sample)
#include "common.cuh"
#include "kernels.h"

namespace gprb {

constexpr int PRED_THREADS = 256;

__device__ __forceinline__ double block_sum(double v, double* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  for (int k = 0; k < PRED_THREADS / 32; ++k) s += red[k];
  return s;
}

// Row chunk i of the split GEMV path covers rows [chunk_begin(i), chunk_begin(i + 1)): row r of L^-1 has r + 1 entries,
// so square-root spacing gives every chunk the same share of V.  Boundaries depend on n only.
__device__ __forceinline__ int chunk_begin(int i, int n) {
  if (i >= PRED_CHUNKS) return n;
  return ((int)((double)n * sqrt((double)i / (double)PRED_CHUNKS))) & ~7;
}

// grid (rsplit, ceil(m / PS), count).  The rows of one (GP, column chunk) are cut into PRED_CHUNKS fixed chunks; the
// `rsplit` CTAs of a (GP, column chunk) take PRED_CHUNKS / rsplit consecutive chunks each, every chunk is reduced by a
// whole CTA in a fixed order and its partial sums go to HBM; the CTA that arrives last adds the partials in chunk order.
// So a single GP with one test column (the reference's call pattern, predictdynamics.jl:13) streams V with 16 CTAs
// instead of one, and the result is bit-identical for every rsplit (i.e. for every batch size).
template <int KIND, int PS>
__global__ void __launch_bounds__(PRED_THREADS) k_predict(PredictArgs g) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* ks = reinterpret_cast<double*>(smem_raw);  // [PS][npad]
  double* xs = ks + (size_t)PS * g.npad;              // [PS][MAX_D]
  double* w = xs + PS * MAX_D;                        // [MAX_D]
  double* red = w + MAX_D;                            // [8]
  __shared__ int is_last;
  const int gl = blockIdx.z, gp = g.gp_off + gl, ci = blockIdx.y, ri = blockIdx.x;
  const int s0 = ci * PS;
  const int ns = min(PS, g.m - s0);
  const int d = g.d, n = g.n, npad = g.npad;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  if (g.mask && g.mask[gp] != 0) {  // no evaluated state: NaN, the other GPs of the call are unaffected
    if (ri == 0 && (int)threadIdx.x < ns) {
      const int64_t o = (int64_t)gl * g.m + s0 + threadIdx.x;
      g.mu[o] = qnan;
      g.var[o] = qnan;
    }
    return;
  }
  const double* th = g.theta + (int64_t)gp * (d + 2);
  const double* Xstar = g.Xstar + (int64_t)(gl / g.gpb) * g.xstar_stride;
  for (int idx = threadIdx.x; idx < PS * d; idx += PRED_THREADS) {
    const int s = idx / d, p = idx % d;
    xs[s * MAX_D + p] = s < ns ? Xstar[(int64_t)(s0 + s) * d + p] : 0.0;
  }
  if (threadIdx.x < d) w[threadIdx.x] = exp(-2.0 * th[1 + threadIdx.x]);
  __syncthreads();
  const double sf2 = exp(2.0 * th[d + 1]);
  const double* X = g.X[gp];
  const double* alpha = g.alpha + (int64_t)gp * npad;
  const int per = PRED_CHUNKS / g.rsplit, ch0 = ri * per, ch1 = ch0 + per;
  const int r_hi = chunk_begin(ch1, n);  // this CTA's rows only meet k*_c for c < r_hi
  for (int r = threadIdx.x; r < r_hi; r += PRED_THREADS) {
    double r2[PS];
#pragma unroll
    for (int s = 0; s < PS; ++s) r2[s] = 0.0;
    const double* xr = X + (int64_t)r * d;
    for (int p = 0; p < d; ++p) {
      const double xv = xr[p], wp = w[p];
#pragma unroll
      for (int s = 0; s < PS; ++s) {
        const double df = xv - xs[s * MAX_D + p];
        r2[s] = fma(wp, df * df, r2[s]);
      }
    }
#pragma unroll
    for (int s = 0; s < PS; ++s) ks[(size_t)s * npad + r] = kcross<KIND>(r2[s], sf2);
  }
  __syncthreads();
  // latent variance through the factor, like the reference's whiten! (PDMats): v = L^-1 k*, var_f = s_f^2 - |v|^2.
  // L^-1 is resident as V = L^-T (strictly-upper tiles of Lm, column r of V = row r of L^-1, contiguous) plus the
  // transposed inverse diagonal blocks DinvT.  Warp per row, lanes over the contiguous column index.
  const double* V = g.Lm + (int64_t)gp * g.mat_stride;
  const double* DT = g.DinvT + (int64_t)gp * g.dinv_stride;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ncc = gridDim.y;
  double* part = g.qpart + ((int64_t)gl * ncc + ci) * (PRED_CHUNKS * 16);
  for (int ch = ch0; ch < ch1; ++ch) {
    const int r0 = chunk_begin(ch, n), r1 = chunk_begin(ch + 1, n);
    double macc[PS], q[PS];
#pragma unroll
    for (int s = 0; s < PS; ++s) macc[s] = q[s] = 0.0;
    for (int r = r0 + threadIdx.x; r < r1; r += PRED_THREADS) {
      const double ar = alpha[r];
#pragma unroll
      for (int s = 0; s < PS; ++s) macc[s] = fma(ks[(size_t)s * npad + r], ar, macc[s]);
    }
    for (int r = r0 + warp; r < r1; r += PRED_THREADS / 32) {
      const int jb = r / NB, rl = r - jb * NB;
      double t[PS];
#pragma unroll
      for (int s = 0; s < PS; ++s) t[s] = 0.0;
      const double* Vr = V + (int64_t)r * npad;
      const int cend = jb * NB;
      for (int c = lane; c < cend; c += 128) {  // four independent loads in flight per lane
        double v[4];
        int cc[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const bool ok = c + 32 * u < cend;
          cc[u] = ok ? c + 32 * u : c;
          v[u] = ok ? Vr[cc[u]] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int s = 0; s < PS; ++s) t[s] = fma(v[u], ks[(size_t)s * npad + cc[u]], t[s]);
      }
      const double* Dr = DT + (int64_t)jb * NB * NB + (int64_t)rl * NB;  // DinvT(c, rl) = inv(L_jj)(rl, c), c <= rl
      for (int c = lane; c <= rl; c += 32) {
        const double v = Dr[c];
#pragma unroll
        for (int s = 0; s < PS; ++s) t[s] = fma(v, ks[(size_t)s * npad + jb * NB + c], t[s]);
      }
#pragma unroll
      for (int s = 0; s < PS; ++s) {
        double v = t[s];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        q[s] = fma(v, v, q[s]);
      }
    }
#pragma unroll
    for (int s = 0; s < PS; ++s) {
      const double mt = block_sum(macc[s], red);
      const double qt = block_sum(lane == 0 ? q[s] : 0.0, red);
      if (threadIdx.x == 0) { part[ch * 16 + s] = mt; part[ch * 16 + 8 + s] = qt; }
    }
  }
  // arrival: the last CTA of this (GP, column chunk) adds the chunk partials in chunk order
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int old = atomicAdd(&g.counter[gl * ncc + ci], 1);
    is_last = (old == g.rsplit - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if ((int)threadIdx.x < ns) {
    const int s = threadIdx.x;
    const volatile double* vp = part;
    double mt = 0.0, qt = 0.0;
    for (int ch = 0; ch < PRED_CHUNKS; ++ch) { mt += vp[ch * 16 + s]; qt += vp[ch * 16 + 8 + s]; }
    const int64_t o = (int64_t)gl * g.m + s0 + s;
    g.mu[o] = mt + (g.mstar ? g.mstar[o] : 0.0);
    g.var[o] = fmax(sf2 - qt, 0.0) + exp(2.0 * th[0]);
  }
  if (threadIdx.x == 0) g.counter[gl * ncc + ci] = 0;
}

// ---------------------------------------------------------------------------------------------------------
// Tiled path (any m, any n): cross-covariance block + mean partials, then L^-1 K* as DMMA tiles (tilegemm.cu,
// GEMM_FWD_ROW) and a finishing reduction.  Follows the reference's whiten! exactly: a forward substitution with
// the factor, no explicit inverse needed, so it also runs on a value-only state (after optimize!).
// ---------------------------------------------------------------------------------------------------------
constexpr int PC_THREADS = 256;

// grid (J, B): CTA = 128 training rows x one chunk of <= 128 test columns of one GP.
// Work unit of a warp = 32 training rows (one per lane) x 8 test columns; ceil(mc / 8) column groups x 4 row blocks per CTA,
// dealt round-robin over the 8 warps (m = 100, the reference's rollout batch: 52 units, 6.5 per warp, 104 of 104 columns
// useful - the lane-per-column layout this replaces computed 128).  Per input dimension a unit costs one conflict-free
// 8-byte load (its row), four broadcast 16-byte loads (the 8 columns) and 16 FP64 instructions, so the FP64 pipe, not the
// shared-memory crossbar, is the limit (the old layout issued one load per 3 FP64 instructions and was crossbar bound).
// Inputs are scaled and centred once in shared memory, z = sqrt(w) (x - x_0) with x_0 the GP's first training sample
// (like k_assemble_gram): r2 = sum (z_i - z_j)^2 is 2 FP64 instructions per pair and dimension instead of 3.
template <int KIND>
__global__ void __launch_bounds__(PC_THREADS) k_predict_cross(PredictTileArgs g) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = g.d;
  double* Xi = reinterpret_cast<double*>(smem_raw);  // [d][NB]   training tile, one row per input dimension
  double* xsT = Xi + d * NB;                          // [d][PT]   test columns, transposed, zero padded
  double* sw = xsT + d * PT;                          // [MAX_D]   sqrt(w_p)
  double* x0 = sw + MAX_D;                            // [MAX_D]   centre
  double* wv = x0 + MAX_D;                            // [MAX_D]   w_p
  double* red = wv + MAX_D;                           // [4][PT]   mean partials per row block
  uint64_t* bar = reinterpret_cast<uint64_t*>(red + 4 * PT);
  const int gl = blockIdx.y, gp = g.gp_off + gl, ib = blockIdx.x;
  if (g.mask && g.mask[gp] != 0) return;  // no evaluated state: k_predict_finish reports NaN
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double* th = g.theta + (int64_t)gp * (d + 2);
  const double* Xt = g.Xt[gp];
  if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_fence_init(); }
  __syncthreads();
  if (threadIdx.x == 0) mbar_expect_tx(bar, (uint32_t)(d * NB * sizeof(double)));
  __syncthreads();
  {  // lane 0 of warps 0-3 issues the copies with warp-uniform operands (per-lane addresses serialise the UBLKCP issue)
    const int uwarp = __shfl_sync(0xffffffffu, warp, 0);
    if (uwarp < 4 && lane == 0)
      for (int p = uwarp; p < d; p += 4) bulk_g2s(Xi + p * NB, Xt + (int64_t)p * g.npad + (int64_t)ib * NB, NB * sizeof(double), bar);
  }
  __shared__ unsigned long long zmax_bits;  // max |z| over the tile and the test columns (bit pattern: non-negative doubles order like integers)
  if (threadIdx.x < d) {
    const double wp = exp(-2.0 * th[1 + threadIdx.x]);
    sw[threadIdx.x] = sqrt(wp);
    wv[threadIdx.x] = wp;
    x0[threadIdx.x] = Xt[(int64_t)threadIdx.x * g.npad];
  }
  if (threadIdx.x == 0) zmax_bits = 0ull;
  __syncthreads();
  const int ncg = (g.mc + 7) >> 3;  // column groups of 8
  const double* Xstar = g.Xstar + (int64_t)(gl / g.gpb) * g.xstar_stride + (int64_t)g.s0 * d;
  double zm = 0.0;
  const int nc8 = 8 * ncg;
  for (int idx = threadIdx.x; idx < d * nc8; idx += PC_THREADS) {
    // consecutive threads walk one input dimension: conflict-free shared-memory stores (the d-strided global reads are a
    // few KB that sit in L2; the transposed order made every store a 32-way bank conflict, 4 us per CTA)
    const int p = idx / nc8, s = idx - p * nc8;
    const double xv = s < g.mc ? Xstar[(int64_t)s * d + p] : x0[p];
    xsT[p * PT + s] = xv;
    zm = fmax(zm, fabs(sw[p] * (xv - x0[p])));
  }
  mbar_wait(bar, 0);
  for (int k = threadIdx.x; k < d * NB; k += PC_THREADS)  // valid rows only: the zero padding behind row n is masked below, whatever it scales to
    if (ib * NB + (k & (NB - 1)) < g.n) zm = fmax(zm, fabs(sw[k >> 7] * (Xi[k] - x0[k >> 7])));
  if (!(zm <= g.zmax)) zm = 1.0e300;  // (also NaN / Inf inputs) -> the unscaled path
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) zm = fmax(zm, __shfl_xor_sync(0xffffffffu, zm, off));
  if (lane == 0) atomicMax(&zmax_bits, (unsigned long long)__double_as_longlong(zm));
  __syncthreads();
  // Scaled path: z = sqrt(w)(x - x_0) rounds every coordinate once, an absolute error of eps |z| in z_i - z_j and so a
  // relative error of <= ~2 eps |z| |z_i - z_j| in K (entries that matter have |z_i - z_j| < 40): below 2e-11 for
  // |z| <= zmax = 1e3.  Extreme length-scales (config.json has l down to 1e-4) keep the raw inputs and the 3-instruction form.
  const bool scaled = __longlong_as_double((long long)zmax_bits) <= g.zmax;
  if (scaled) {
    for (int idx = threadIdx.x; idx < d * nc8; idx += PC_THREADS) {
      const int p = idx / nc8, s = idx - p * nc8;
      xsT[p * PT + s] = sw[p] * (xsT[p * PT + s] - x0[p]);
    }
    for (int k = threadIdx.x; k < d * NB; k += PC_THREADS) Xi[k] = sw[k >> 7] * (Xi[k] - x0[k >> 7]);
    __syncthreads();
  }
  const double sf2 = exp(2.0 * th[d + 1]);
  const double* alpha = g.alpha + (int64_t)gp * g.npad;
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
  for (int u = warp; u < 4 * ncg; u += PC_THREADS / 32) {
    const int cg = u >> 2, rb = u & 3, rl = rb * 32 + lane, r = ib * NB + rl;
    double r2[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r2[k] = 0.0;
    const double* xr = Xi + rl;
    const double* xc = xsT + 8 * cg;
    if (scaled) {
#pragma unroll 2
      for (int p = 0; p < d; ++p) {
        const double xv = xr[p * NB];
        const double2* cp = reinterpret_cast<const double2*>(xc + p * PT);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const double2 c = cp[k];
          const double d0 = xv - c.x, d1 = xv - c.y;
          r2[2 * k] = fma(d0, d0, r2[2 * k]);
          r2[2 * k + 1] = fma(d1, d1, r2[2 * k + 1]);
        }
      }
    } else {
      for (int p = 0; p < d; ++p) {
        const double xv = xr[p * NB], wp = wv[p];
        const double2* cp = reinterpret_cast<const double2*>(xc + p * PT);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const double2 c = cp[k];
          const double d0 = xv - c.x, d1 = xv - c.y;
          r2[2 * k] = fma(wp, d0 * d0, r2[2 * k]);
          r2[2 * k + 1] = fma(wp, d1 * d1, r2[2 * k + 1]);
        }
      }
    }
    const bool rok = r < g.n;
    const double ar = rok ? alpha[r] : 0.0;
    double v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = (rok && 8 * cg + k < g.mc) ? kcross<KIND>(r2[k], sf2) : 0.0;
    if (g.T) {
      double2* tp = reinterpret_cast<double2*>(g.T + ((int64_t)gl * g.npad + r) * PT + 8 * cg);
#pragma unroll
      for (int k = 0; k < 4; ++k) tp[k] = make_double2(v[2 * k], v[2 * k + 1]);
    }
    // mean partials: sum over the 32 rows of v[k] alpha_r for the 8 columns - a transposing butterfly (4 + 2 + 1 exchanges
    // halve the values a lane carries, two more finish the sum): 9 shuffles instead of 40, fixed order
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] *= ar;
    double a4[4], a2[2];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double send = b4 ? v[k] : v[k + 4], keep = b4 ? v[k + 4] : v[k];
      a4[k] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const double send = b3 ? a4[k] : a4[k + 2], keep = b3 ? a4[k + 2] : a4[k];
      a2[k] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    double a1 = (b2 ? a2[1] : a2[0]) + __shfl_xor_sync(0xffffffffu, b2 ? a2[0] : a2[1], 4);
    a1 += __shfl_xor_sync(0xffffffffu, a1, 2);
    a1 += __shfl_xor_sync(0xffffffffu, a1, 1);
    if ((lane & 3) == 0) red[rb * PT + 8 * cg + (b4 ? 4 : 0) + (b3 ? 2 : 0) + (b2 ? 1 : 0)] = a1;
  }
  __syncthreads();
  if ((int)threadIdx.x < 8 * ncg)
    g.mupart[((int64_t)gl * g.J + ib) * PT + threadIdx.x] = (red[threadIdx.x] + red[PT + threadIdx.x]) + (red[2 * PT + threadIdx.x] + red[3 * PT + threadIdx.x]);
}

// grid B, 512 threads: thread = (row partition, test column).  mu = sum of the block partials + m(x*);
// var = max(s_f^2 - sum_r T(r,s)^2, 0) + exp(2 logNoise), fixed summation order.
__global__ void __launch_bounds__(512) k_predict_finish(PredictTileArgs g) {
  __shared__ double red[4][PT];
  const int gl = blockIdx.x, gp = g.gp_off + gl, s = threadIdx.x & (PT - 1), part = threadIdx.x >> 7;
  const int d = g.d;
  const double* th = g.theta + (int64_t)gp * (d + 2);
  if (g.mask && g.mask[gp] != 0) {  // no evaluated state: NaN rows, the other GPs of the call are unaffected
    if (part == 0 && s < g.mc) {
      const int64_t o = (int64_t)gl * g.m + g.s0 + s;
      g.mu[o] = __longlong_as_double(0x7ff8000000000000LL);
      if (g.var) g.var[o] = __longlong_as_double(0x7ff8000000000000LL);
    }
    return;
  }
  if (g.var && s < g.mc) {  // the columns beyond mc of a chunk are never read (k_predict_cross does not write them either)
    const double* T = g.T + (int64_t)gl * g.npad * PT + s;
    const int per = (g.n + 3) / 4, r0 = part * per, r1 = min(g.n, r0 + per);
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int r = r0;
    for (; r + 7 < r1; r += 8) {  // eight loads in flight per thread; every accumulator still sees its rows in the same order
      const double v0 = T[(int64_t)r * PT], v1 = T[(int64_t)(r + 1) * PT], v2 = T[(int64_t)(r + 2) * PT], v3 = T[(int64_t)(r + 3) * PT];
      const double v4 = T[(int64_t)(r + 4) * PT], v5 = T[(int64_t)(r + 5) * PT], v6 = T[(int64_t)(r + 6) * PT], v7 = T[(int64_t)(r + 7) * PT];
      a0 = fma(v0, v0, a0); a1 = fma(v1, v1, a1); a2 = fma(v2, v2, a2); a3 = fma(v3, v3, a3);
      a0 = fma(v4, v4, a0); a1 = fma(v5, v5, a1); a2 = fma(v6, v6, a2); a3 = fma(v7, v7, a3);
    }
    for (; r + 3 < r1; r += 4) {
      const double v0 = T[(int64_t)r * PT], v1 = T[(int64_t)(r + 1) * PT], v2 = T[(int64_t)(r + 2) * PT], v3 = T[(int64_t)(r + 3) * PT];
      a0 = fma(v0, v0, a0); a1 = fma(v1, v1, a1); a2 = fma(v2, v2, a2); a3 = fma(v3, v3, a3);
    }
    for (; r < r1; ++r) { const double v = T[(int64_t)r * PT]; a0 = fma(v, v, a0); }
    red[part][s] = (a0 + a1) + (a2 + a3);
  }
  __syncthreads();
  if (part != 0 || s >= g.mc) return;
  const int64_t o = (int64_t)gl * g.m + g.s0 + s;
  double mu = 0.0;
  for (int ib = 0; ib < g.J; ++ib) mu += g.mupart[((int64_t)gl * g.J + ib) * PT + s];
  g.mu[o] = mu + (g.mstar ? g.mstar[o] : 0.0);
  if (g.var) {
    const double q = (red[0][s] + red[1][s]) + (red[2][s] + red[3][s]);
    g.var[o] = fmax(exp(2.0 * th[d + 1]) - q, 0.0) + exp(2.0 * th[0]);
  }
}

int launch_predict_cross(const PredictTileArgs& a, int count, cudaStream_t stream) {
  const int B = count;
  if (B <= 0 || a.mc <= 0) return 0;
  const size_t smem = ((size_t)a.d * NB + (size_t)a.d * PT + 3 * MAX_D + 4 * PT) * sizeof(double) + 16;
  dim3 grid(a.J, B);
  cudaError_t e;
#define GPRB_PC_CASE(K)                                                                                       \
  e = cudaFuncSetAttribute(k_predict_cross<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);       \
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_predict_cross)", __FILE__, __LINE__);     \
  k_predict_cross<K><<<grid, PC_THREADS, smem, stream>>>(a);
  switch (a.kind) {
    case GPRB_KERNEL_SE_ARD: GPRB_PC_CASE(0) break;
    case GPRB_KERNEL_MAT12_ARD: GPRB_PC_CASE(1) break;
    case GPRB_KERNEL_MAT32_ARD: GPRB_PC_CASE(2) break;
    default: GPRB_PC_CASE(3) break;
  }
#undef GPRB_PC_CASE
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_predict_cross launch", __FILE__, __LINE__);
  return 0;
}

int launch_predict_finish(const PredictTileArgs& a, int count, cudaStream_t stream) {
  const int B = count;
  if (B <= 0 || a.mc <= 0) return 0;
  k_predict_finish<<<B, 512, 0, stream>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_predict_finish launch", __FILE__, __LINE__);
  return 0;
}

int launch_predict(const PredictArgs& a, int count, cudaStream_t stream) {
  if (count <= 0 || a.m <= 0) return 0;
  const int ps = a.m <= 1 ? 1 : a.m <= 2 ? 2 : a.m <= 4 ? 4 : 8;  // test columns per CTA (smem: ps * npad doubles)
  const size_t smem = ((size_t)ps * a.npad + ps * MAX_D + MAX_D + 8) * sizeof(double);
  if (smem > 227 * 1024) {
    set_error("gprb_predict: n too large for the shared-memory cross-covariance block");
    return GPRB_ERR_ARG;
  }
  dim3 grid(a.rsplit, (a.m + ps - 1) / ps, count);
  cudaError_t e;
#define GPRB_PRED_LAUNCH(K, P)                                                                                 \
  e = cudaFuncSetAttribute(k_predict<K, P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);            \
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_predict)", __FILE__, __LINE__);            \
  k_predict<K, P><<<grid, PRED_THREADS, smem, stream>>>(a);
#define GPRB_PRED_CASE(K)                                   \
  if (ps == 1) { GPRB_PRED_LAUNCH(K, 1) }                   \
  else if (ps == 2) { GPRB_PRED_LAUNCH(K, 2) }              \
  else if (ps == 4) { GPRB_PRED_LAUNCH(K, 4) }              \
  else { GPRB_PRED_LAUNCH(K, 8) }
  switch (a.kind) {
    case GPRB_KERNEL_SE_ARD: GPRB_PRED_CASE(0) break;
    case GPRB_KERNEL_MAT12_ARD: GPRB_PRED_CASE(1) break;
    case GPRB_KERNEL_MAT32_ARD: GPRB_PRED_CASE(2) break;
    default: GPRB_PRED_CASE(3) break;
  }
#undef GPRB_PRED_CASE
#undef GPRB_PRED_LAUNCH
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_predict launch", __FILE__, __LINE__);
  return 0;
}

}  // namespace gprb
