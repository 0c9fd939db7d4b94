// Launcher prototypes of the libgprb200 CUDA stages (host-callable, defined in the .cu files).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace gprb {

enum { GEMM_CHOL_DIAG = 0, GEMM_CHOL_COL = 1, GEMM_TRTRI_ROW = 2, GEMM_LAUUM = 3, GEMM_FWD_ROW = 4,
       GEMM_CHOL_PANEL = 5, GEMM_CHOL_TRAIL = 6,   // right-looking Cholesky for small batches (latency-bound chains)
       GEMM_BWD_ROW = 7 };                         // backward substitution L^-T T of the predictive gradient (k_tile_bwd)

struct GemmArgs {
  const double* Lm;     // operand matrices [B][npad*npad]
  const double* DinvT;  // transposed inverse diagonal blocks [B][J][NB*NB] (operand substitute for V(k,k))
  const double* Dinv;   // inverse diagonal blocks (post-multiplier)
  const double* Cin;    // K tiles for the Cholesky modes
  double* Cout;
  double* KinvD;        // [B][J][NB*NB] diagonal tiles of K^-1 (LAUUM output)
  const int32_t* list;  // GP index per blockIdx.y (nullptr = identity)
  int64_t mat_stride, dinv_stride;
  int npad, J, step, mode;
  int nv;               // n rounded up to 16: rows / k beyond it are padding that is neither computed nor read
  int row0 = 0;         // GEMM_CHOL_COL: first block row of the launch, i = max(step + 1, row0) + blockIdx (gprb_batch_append
                        // refactorises only the block rows its new samples reach)
  // GEMM_FWD_ROW only: the right-hand-side block T [B][npad][ldt] (row r of T contiguous over the test columns);
  // it is the B operand, the Cin source and the output at once (block row `step` is solved in place)
  double* Tm = nullptr;
  int64_t t_stride = 0;
  int ldt = 0;
  int ncols = 128;      // valid test columns of the block (< 128: compact warp layout skips the padding columns)
  int colw = 64;        // columns per FWD_ROW tile (64 or 32): tile bx owns columns bx*colw .. of the block
  int gp_off = 0;       // first GP of this launch when `list` is null (stream groups of gprb_predict)
  int t_gp_off = 0;     // GEMM_FWD_ROW: Tm is indexed by gp - t_gp_off (the right-hand-side blocks of a GP range start at its first GP)
  const int32_t* fail = nullptr;     // [B] per-GP failure flag: tiles of a GP whose factorisation already broke down exit at once
  unsigned long long* tl = nullptr;  // debug timeline buffer [count][ntiles][8] (only read when built with -DGPRB_TIMELINE)
  // TMA tensor maps of the operands (gprb_batch / gprb_predict_slot own them): box = 132 or 68 padded rows x KT columns
  CUtensorMap tm_L132, tm_L68, tm_DT132, tm_DT68, tm_D132, tm_T68, tm_A68;
  int pf_cin = 0;       // 1: Cin is the matrix tm_A68 describes - the CTA prefetches its K half tile into L2 with TMA requests at entry
  CUtensorMap tm_LT;    // GEMM_BWD_ROW only: Lm with box = KT rows x NB columns (L(k, i)^T lands row-major)
};

int launch_tile_gemm(const GemmArgs& g, int ntiles, int count, cudaStream_t stream);
int configure_tile_gemm();    // per-device shared-memory opt-in (current device); called by gprb_init

// K1: covariance assembly, lower tiles of K = K_f + (exp(2 logNoise) + eps + jitter) I ; identity in the padding.
struct AssembleArgs {
  const double* const* Xt;  // [B] per-GP pointer to the dataset's transposed inputs Xt[d][npad]
  const double* theta;      // [B][P]
  const double* jitter;     // [B]
  double* A;                // [B][npad*npad]
  double* A2 = nullptr;     // optional second copy of the lower tiles (the right-looking factorisation works in place in Lm)
  int32_t* fail;            // [B] reset here: 0, or -2 for non-finite theta
  const int32_t* list;
  int64_t mat_stride;
  int n, npad, d, J, kind;
  int tile0 = 0;            // first lower tile (row-by-row order) of the launch: j0 (j0 + 1) / 2 assembles block rows >= j0 only
};
int launch_assemble(const AssembleArgs& a, int count, cudaStream_t stream);

// potf2 + trtri of the 128x128 diagonal block `step` (in place in Lm), emits Dinv, DinvT, logdet partials, fail flag.
struct DiagArgs {
  const double* Src = nullptr;  // where the block to factorise is read from (nullptr = Lm): block column 0 has no update
                                // terms, so its diagonal block is taken straight from K (no CHOL_DIAG copy launch)
  double* Lm;
  double* Dinv;
  double* DinvT;
  double* logdet_part;  // [B][J]
  int32_t* fail;        // [B]
  const int32_t* list;
  int64_t mat_stride, dinv_stride;
  int npad, J, step;
  int nv;
};
int launch_diag_factor(const DiagArgs& a, int count, cudaStream_t stream);
int configure_diag_factor();  // per-device shared-memory opt-in (current device); called by gprb_init

// forward + backward substitution, alpha = K^-1 ymm, and mll = -1/2 (ymm'alpha + logdet + n log 2pi).
struct SolveArgs {
  const double* Lm;
  const double* Dinv;
  const double* ymm;          // [B][npad]
  const double* logdet_part;  // [B][J]
  const int32_t* fail;
  double* zbuf;               // [B][npad]
  double* alpha;              // [B][npad]
  double* mll;                // [B]
  const int32_t* list;
  int64_t mat_stride, dinv_stride;
  int n, npad, J;
  int nv;
  int cluster_below = 0;      // passes with fewer GPs than this run one thread-block cluster per GP (k_solve_cluster)
};
int launch_solve(const SolveArgs& a, int count, cudaStream_t stream);

constexpr int GRAD_PARTS_PER_TILE = 4;  // k_grad_tiles splits every 128x128 tile into 128 x 32 column blocks (one CTA each)
// K5: fused gradient  d mll / d theta = 1/2 tr((alpha alpha' - K^-1) dK/dtheta), never materialising dK.
struct GradArgs {
  const double* const* Xt;
  const double* theta;
  const double* A;      // lower tiles: K (intact); strictly-upper tile (j,i): K^-1 tile (i,j), un-transposed
  const double* KinvD;  // [B][J][NB*NB] diagonal tiles of K^-1
  const double* alpha;
  double* part;         // [B][ntiles * GRAD_PARTS_PER_TILE][P]
  double* grad;         // [B][P]
  const int32_t* fail;
  const int32_t* list;
  int64_t mat_stride, dinv_stride;
  int n, npad, d, J, kind;
};
int launch_grad(const GradArgs& a, int count, cudaStream_t stream);

// dataset helpers
int launch_transpose_inputs(const double* X, double* Xt, int n, int npad, int d, cudaStream_t stream);
int launch_transpose_inputs_batched(const double* X, double* Xt, int n, int npad, int d, int count, cudaStream_t stream);
// jitter[gp] += 1e-6 * tr(K)/n for the listed GPs (make_posdef!); applied by the next assembly
int launch_add_jitter(const double* theta, double* jitter, const int32_t* list, int d, int count, cudaStream_t stream);

// K6: posterior mean / variance
// GPs gp_off .. gp_off + count - 1 of the batch; Xstar / mstar / mu / var / scratch are indexed by the LOCAL GP index
// (gp - gp_off), theta / alpha / Lm / X by the global one.  mask[gp] != 0: no evaluated state, outputs NaN.
constexpr int PRED_CHUNKS = 16;  // fixed row chunks of the split GEMV path (partials are summed in chunk order: results
                                 // do not depend on how many CTAs share the chunks, i.e. on the batch size)
struct PredictArgs {
  const double* const* X;  // [B] original d x n inputs
  const double* theta;
  const double* alpha;
  const double* Lm;        // V = L^-T in the strictly-upper tiles (variance only)
  const double* DinvT;     // transposed inverse diagonal blocks
  const double* Xstar;     // d x m (+ local gp * xstar_stride)
  const double* mstar;     // [count][m] or nullptr
  double* mu;              // [count][m]
  double* var;             // [count][m]
  double* qpart;           // [count][colchunks][PRED_CHUNKS][2][8] partial mean / |L^-1 k*|^2 sums
  int32_t* counter;        // [count * colchunks] arrival counters (zero on entry, reset by the last CTA)
  const int32_t* mask;     // [B]
  int64_t xstar_stride, mat_stride, dinv_stride;
  int n, npad, d, m, kind;
  int gp_off, rsplit;      // rsplit in {1, 2, 4, 8, 16}: CTAs sharing the PRED_CHUNKS row chunks of one (GP, column chunk)
  int gpb = 1;             // consecutive GPs sharing one Xstar block (the G outputs of a trial): block = local gp / gpb
};
int launch_predict(const PredictArgs& a, int count, cudaStream_t stream);  // small-m path (needs V resident)

// Tiled path: cross-covariances of one chunk of <= 128 test columns -> T[B][npad][PT] (+ per-block mean partials),
// then the forward substitution L^-1 K* runs as GEMM_FWD_ROW launches and k_predict_finish reduces.
constexpr int PT = 128;  // test columns per chunk (row length of T)
struct PredictTileArgs {
  const double* const* Xt;  // [B] transposed training inputs Xt[d][npad]
  const double* theta;
  const double* alpha;
  const double* Xstar;      // d x m (+ b * xstar_stride)
  const double* mstar;      // [B][m] or nullptr
  double* T;                // [count][npad][PT] or nullptr (mean only)
  double* mupart;           // [count][J][PT]
  double* mu;               // [count][m]
  double* var;              // [count][m] or nullptr
  int64_t xstar_stride;
  int n, npad, d, J, m, kind;
  int s0, mc;               // chunk: test columns s0 .. s0 + mc
  int gp_off = 0;           // first GP of the range (local index = gp - gp_off, see PredictArgs)
  const int32_t* mask = nullptr;  // [B] or nullptr
  int gpb = 1;              // consecutive GPs sharing one Xstar block (see PredictArgs)
  double zmax = 1.0e3;      // largest scaled, centred input coordinate k_predict_cross uses its 2-instruction distance form for
};
int launch_predict_cross(const PredictTileArgs& a, int count, cudaStream_t stream);
int launch_predict_finish(const PredictTileArgs& a, int count, cudaStream_t stream);

// Predictive gradients (predgrad.cu): dmu / dx* = dm(x*) + sum_i alpha_i dk(x*, x_i) / dx* and
// dvar / dx* = -2 sum_i beta_i dk(x*, x_i) / dx*, beta = L^-T L^-1 K* (the T block after the FWD_ROW and BWD_ROW chains),
// for one chunk of <= PT test columns.  One CTA per GP; blockIdx.x = gp - gp_off like k_predict_finish.
struct PredictJacArgs {
  const double* const* Xt;  // [B] transposed training inputs Xt[d][npad]
  const double* theta;
  const double* alpha;
  const double* beta;       // [count][npad][PT] or nullptr (mean only)
  const double* Xstar;      // d x m (+ local gp * xstar_stride)
  const double* dmstar;     // [count][m][d] or nullptr
  double* dmu;              // [count][m][d]
  double* dvar;             // [count][m][d] or nullptr
  const int32_t* mask;      // [B]
  int64_t xstar_stride;
  int n, npad, d, m, kind;
  int s0, mc;               // chunk: test columns s0 .. s0 + mc
  int gp_off;
};
int launch_predict_jac(const PredictJacArgs& a, int count, cudaStream_t stream);

// Full posterior covariance (postcov.cu): Sigma = K** - T'T (+ exp(2 logNoise) I) from the solved right-hand sides
// T = L^-1 K* of every 128-column chunk, one CTA per lower 128 x 128 tile of Sigma and GP, both triangles written.
// GPs gp_off .. gp_off + count - 1; T / S / bad are indexed by the local GP index (gp - gp_off) like PredictTileArgs.
constexpr int POSTCOV_MAX_M = 8192;
struct PostCovArgs {
  const double* Xstar;  // d x m (+ local gp * xstar_stride)
  const double* theta;
  const int32_t* mask;  // [B]: 1 = no evaluated state (Sigma rows come back NaN)
  double* S;            // [nloc][mpad][mpad] column-major; rows / columns >= m are the identity
  int32_t* bad;         // [nloc] or nullptr: set to 1 when the GP's Sigma holds a non-finite entry
  int64_t xstar_stride;
  int nv, d, m, mpad, kind;
  int gp_off, nloc;     // nloc: GPs of the whole call (chunk c of local GP g is GP index c * nloc + g of tm_T68)
  int g0;               // first local GP of this launch (a stream group of the call): blockIdx.y + g0 = local GP
  int add_noise;
  CUtensorMap tm_T68;   // the T blocks [chunk][nloc][npad][PT], box = 68 test columns x KT rows (the GEMM_FWD_ROW map)
};
int launch_post_cov(const PostCovArgs& a, int count, cudaStream_t stream);
int configure_post_cov();  // per-device shared-memory opt-in (current device); called by gprb_init

// make_posdef! on Sigma_f of the listed GPs: A_ii += 1e-6 tr(A)/m (i < m, fixed summation order), fail reset to 0
int launch_post_jitter(double* S, int32_t* fail, const int32_t* list, int m, int mpad, int count, cudaStream_t stream);
// fail[g] = -2 for GPs without state (mask[gp_off + g]) or with a non-finite Sigma (bad[g]), else 0
int launch_post_fail_init(int32_t* fail, const int32_t* mask, const int32_t* bad, int gp_off, int count, cudaStream_t stream);
// out[g][s][i] = mu[g][i] + sum_{k <= i} L(i,k) Z[g][s][k] (k ascending); NaN for the GPs with fail[g] != 0
struct PostDrawArgs {
  const double* L;     // [count][mpad][mpad] lower factor (column-major)
  const double* mu;    // [count][m]
  const double* Z;     // [count][ns][m]
  const int32_t* fail;
  double* out;         // [count][ns][m]
  int m, mpad, ns;
};
int launch_post_draws(const PostDrawArgs& a, int count, cudaStream_t stream);

// Leave-one-out cross-validation (loo.cu), Rasmussen & Williams eqs. 5.10-5.13 on the resident K^-1 and alpha, for the
// GPs gp0 .. gp0 + cnt - 1.  Batch buffers (A, KinvD, alpha, ymm, skip, mu, var, logp) are indexed by the global GP
// index, the per-call workspace (v, s, u, G, W, Ap, KinvDp) by the local one (gp - gp0).  skip[gp] != 0: not processed.
struct LooArgs {
  const double* A;       // batch [B][npad*npad]: K in the lower tiles, K^-1 tile (i,j), i > j, at tile position (j,i)
  const double* KinvD;   // batch [B][J][NB*NB] diagonal tiles of K^-1
  const double* alpha;   // batch [B][npad]
  const double* ymm;     // batch [B][npad]
  const int32_t* skip;   // [B]
  double* v;             // [cnt][npad] alpha ./ diag(K^-1), zero padded (nullptr: value only)
  double* s;             // [cnt][npad] sqrt(-c), c_i = -1/2 (1 + alpha_i^2 / d_i) / d_i, zero padded
  const double* u;       // [cnt][npad] K^-1 v
  double* G;             // [J][cnt][npad][PT] diag(s) K^-1 in the right-hand-side layout of GEMM_FWD_ROW / k_post_cov
  const double* W;       // [cnt][npad][npad] K^-1 diag(c) K^-1, exactly symmetric
  double* Ap;            // [cnt][npad][npad] K in the lower tiles, -Q' in the strictly-upper ones (K^-1 convention)
  double* KinvDp;        // [cnt][J][NB*NB] diagonal tiles of -Q'
  double* mu;            // [B][n] y - m(X) - alpha_i / d_i
  double* var;           // [B][n] 1 / d_i
  double* logp;          // [B]
  int64_t mat_stride, dinv_stride;
  int n, npad, J, gp0;
};
int launch_loo_point(const LooArgs& a, int count, cudaStream_t stream);     // pointwise terms, logp, v and s
int launch_loo_expand(const LooArgs& a, int count, cudaStream_t stream);    // G = diag(s) K^-1
int launch_loo_assemble(const LooArgs& a, int count, cudaStream_t stream);  // Ap, KinvDp
// W = -G'G on the DMMA pipe: k_post_cov with zero-initialised accumulators (no K** prologue, no noise), m = n, mpad = npad
int launch_loo_w(const PostCovArgs& a, int count, cudaStream_t stream);

}  // namespace gprb
