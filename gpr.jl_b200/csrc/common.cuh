// Shared definitions for libgprb200: handles, launch geometry, sm_100a PTX helpers.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/gprb200.h"
#include "kernels.h"

namespace gprb {

constexpr int NB = 128;        // tile edge of every blocked fp64 stage (Cholesky / TRTRI / LAUUM)
constexpr int KT = 16;         // k-extent of one pipeline stage of the tile GEMM
constexpr int LDS_T = NB + 4;  // padded smem row (doubles): (t*132 + g) mod 16 distinct over a half-warp
constexpr int MAX_D = 62;      // 13 * bodies <= 52 in the reference (src/CState.jl:20); (MAX_D + 2) * 128 doubles fit the
                               // 64 KB landing zone the gradient kernel reuses as its reduction buffer
constexpr int MAX_JITTER = 10; // make_posdef! retries (GaussianProcesses 0.12.4)
constexpr int MAX_STREAMS = 8; // the GPs of one call are split over up to this many streams (GPRB200_STREAMS, default 4);
                               // prediction slot s owns stream[4s .. 4s+3]

void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

// TMA tensor map over a batched column-major fp64 array viewed as [dim2 = GP][dim1 = column][dim0 = row]:
// one cp.async.bulk.tensor request (SASS UTMALDG) then lands a whole k-chunk of `box_cols` columns x `box_rows` rows in
// shared memory.  box_rows is the PADDED row count (132 / 68 for 128- / 64-row operands): the box simply reads 4 rows
// more than the operand needs (zero-filled where that leaves the array), which makes the smem pitch equal to the
// bank-conflict-free padded pitch of the DMMA fragment loads - a tiled box has no pitch of its own.
int make_tensor_map(CUtensorMap* map, const double* base, uint64_t rows, uint64_t cols, uint64_t gps, uint64_t col_stride_doubles,
                    uint64_t gp_stride_doubles, uint32_t box_rows, uint32_t box_cols);

#define GPRB_CUDA(call)                                                        \
  do {                                                                         \
    cudaError_t e__ = (call);                                                  \
    if (e__ != cudaSuccess) return ::gprb::cuda_fail(e__, #call, __FILE__, __LINE__); \
  } while (0)

#define GPRB_REQUIRE(cond, msg)          \
  do {                                   \
    if (!(cond)) {                       \
      ::gprb::set_error(msg);            \
      return GPRB_ERR_ARG;               \
    }                                    \
  } while (0)

// One evaluation pass for the batched optimiser (api.cu): like gprb_eval_mixed, but the make_posdef! retries are NOT
// looped inside - a GP whose factorisation failed comes back with pending[gp] = 1 and is re-submitted (retry[gp] = 1,
// same theta, one more jitter) together with the next round's evaluations of the other GPs.
int eval_pass_host(gprb_batch* b, const double* theta, const uint8_t* mode, const uint8_t* retry, double* mll, double* grad,
                   int32_t* info, uint8_t* pending);

// GPRB_ERR_ARG with "<fn>: a prediction is in flight - call gprb_predict_wait first" while either prediction slot of b
// is pending, 0 otherwise: the calls that write a batch's resident state (theta, K, factor, alpha, targets, offsets)
// refuse then, because the slots' streams are not ordered with the evaluation streams.
int refuse_while_predicting(const gprb_batch* b, const char* fn);

}  // namespace gprb

struct gprb_ctx;
namespace gprb {
void comm_release(gprb_ctx* ctx);  // comm.cu: destroy the context's NCCL communicator and gather staging
}

struct gprb_ctx {
  int device = 0;
  int sm_count = 0;
  int clock_khz = 0;
  int64_t l2_bytes = 0;
  int64_t launches = 0;
  cudaStream_t upload = nullptr;   // dataset uploads (non-blocking stream)
  cudaStream_t upload2 = nullptr;  // input transposes of a batched upload, behind upload_ev
  cudaEvent_t upload_ev = nullptr;
  // final gather (comm.cu): NCCL communicator of this context's rank, grow-only device / pinned staging
  void* comm = nullptr;            // ncclComm_t
  int rank = 0, nranks = 1;
  double* gather_dev = nullptr;    // [send | recv]
  double* gather_host = nullptr;   // pinned, same layout
  size_t gather_cap = 0;           // doubles
};

// One device allocation shared by the datasets of gprb_datasets_create (freed with the last member).
struct gprb_slab {
  double* X = nullptr;   // [count][d*n]
  double* Xt = nullptr;  // [count][d*npad]
  int32_t count = 0;
  int32_t refs = 0;
};

struct gprb_dataset {
  gprb_ctx* ctx = nullptr;
  int64_t n = 0;
  int32_t d = 0;
  int64_t npad = 0;      // n rounded up to a multiple of NB
  double* X = nullptr;   // device, d x n column-major (sample = contiguous column), tightly packed
  double* Xt = nullptr;  // device, Xt[p][npad]: one contiguous, zero-padded row per input dimension (TMA source)
  uint64_t version = 0;  // bumped by every upload (state reuse compares it)
  gprb_slab* slab = nullptr;  // non-null: X / Xt point into the slab (member `slab_index`)
  int32_t slab_index = 0;
  int32_t users = 0;     // live batches that use the dataset (gprb_batch_append grows only a dataset no other batch reads)
  int32_t predicting = 0;  // predictions in flight (gprb_predict_async, not yet waited for) that read X / Xt: uploads refuse
};

// One prediction pipeline of a batch (gprb_predict_async slot): own streams, staging and scratch, so that two groups
// of trials can be in flight at once (device predict of one group under the host projection of the other).
struct gprb_predict_slot {
  double* pX = nullptr; double* pms = nullptr; double* pmu = nullptr; double* pvar = nullptr;  // device
  double* pT = nullptr; double* pmupart = nullptr; double* pq = nullptr;
  CUtensorMap tm_T68;          // pT [count][npad][PT], re-encoded whenever pT is (re)allocated
  size_t tm_T_cap = 0;
  int32_t* pcount = nullptr;   // [cap_gps] arrival counters of the split GEMV path (zero between calls)
  int32_t* mask = nullptr;     // device [B]: 1 = GP has no evaluated state (outputs NaN)
  size_t pX_cap = 0, pms_cap = 0, pmu_cap = 0, pvar_cap = 0, pT_cap = 0, pmupart_cap = 0, pq_cap = 0, pcount_cap = 0;
  double* h_in = nullptr; double* h_out = nullptr;  // pinned staging: [Xstar | mstar] and [mu | var]
  int32_t* h_mask = nullptr;                        // pinned [B]
  size_t h_in_cap = 0, h_out_cap = 0;
  cudaEvent_t t0 = nullptr, t1 = nullptr;           // device time of the last prediction
  bool pending = false;
  std::vector<gprb_dataset*> reads;  // distinct datasets of GPs gp0 .. gp1-1 while pending (their `predicting` is raised)
  int gp0 = 0, gp1 = 0;
  int64_t m = 0;
  bool want_var = false;
  double last_ms = 0.0;
};

// Workspace of gprb_predict_cov / gprb_sample_posterior (allocated on first use, grow-only; slot 0's streams, staging and
// events run the calls).  mpad = m rounded up to NB, Jm = mpad / NB.
struct gprb_postcov_ws {
  double* T = nullptr;      // [chunk][B][npad][PT] right-hand sides L^-1 K* of every 128-column chunk
  double* S = nullptr;      // [B][mpad][mpad] Sigma (identity padding); the make_posdef! jitter is added in place
  double* L = nullptr;      // [B][mpad][mpad] lower factor of Sigma_f
  double* Dinv = nullptr; double* DinvT = nullptr;  // [B][Jm][NB*NB]; the structural-zero halves are set at allocation
  double* logdet = nullptr; // [B][Jm] (written by k_diag_factor, unused)
  double* Z = nullptr;      // [B][ns][m] standard normals
  double* O = nullptr;      // [B][m][m] packed Sigma / [B][ns][m] draws for the copy to the host
  int32_t* bad = nullptr;   // [B] 1 = non-finite Sigma
  int32_t* fail = nullptr;  // [B] factorisation status (LAPACK info, -2 no state / non-finite)
  int32_t* list = nullptr;  // [B] GPs of a make_posdef! retry
  int32_t* fail_host = nullptr; int32_t* list_host = nullptr;  // pinned [B]
  size_t T_cap = 0, S_cap = 0, L_cap = 0, D_cap = 0, logdet_cap = 0, Z_cap = 0, O_cap = 0, bad_cap = 0, fail_cap = 0, list_cap = 0;
  CUtensorMap tm_T68;       // T as [chunk * B + GP][npad][PT], box = 68 test columns x KT rows (GEMM_FWD_ROW and k_post_cov)
  cudaEvent_t z_ready = nullptr;  // Z has arrived (its copy runs on the upload stream, under the T solve)
};

// Workspace of gprb_eval_loo (allocated on first use, grow-only).  The GPs are processed in groups of at most `cap`
// consecutive batch indices; the group buffers are indexed by the GP's position in its group.
struct gprb_loo_ws {
  double* M = nullptr;      // [cap][npad][npad] G = diag(sqrt(-c)) K^-1 (chunked right-hand-side layout), then A'
  double* W = nullptr;      // [cap][npad][npad] K^-1 diag(c) K^-1
  double* KD = nullptr;     // [cap][J][NB*NB] diagonal tiles of -Q'
  double* vec = nullptr;    // [5][cap][npad] v = alpha ./ d, s = sqrt(-c), u = K^-1 v, the substitution's z, zero alpha
  double* part = nullptr;   // [cap][ntiles * GRAD_PARTS_PER_TILE][P] gradient partial sums
  double* mll = nullptr;    // [cap] the substitution's mll (not used)
  int cap = 0;              // GPs per group the buffers above hold
  double* out = nullptr;    // logp [B] | grad [B][P] | mu [B][n] | var [B][n], indexed by the batch GP index
  int32_t* skip = nullptr;  // [B] 1 = not processed (inactive or failed evaluation)
  int32_t* skip_host = nullptr;  // pinned [B]
  size_t out_cap = 0;
};

// Workspace of gprb_predict_grad (allocated on first use, grow-only; slot 0's streams, staging, T block and events run the
// call).  Only the outputs grow with m: the right-hand sides are one 128-column chunk per GP (the slot's pT).
struct gprb_predgrad_ws {
  double* jac = nullptr;    // [2][B][m][d] dmu | dvar
  double* dms = nullptr;    // [B][m][d] prior-mean Jacobian
  size_t jac_cap = 0, dms_cap = 0;
};

// Per-GP device state (structure-of-arrays over the batch), all resident in HBM:
//   A   [B][npad*npad]  K in the lower tiles (kept); after the inverse stage the strictly-upper tile (j,i) holds the
//                       K^-1 tile (i,j) un-transposed, and KinvD the diagonal tiles of K^-1
//   Lm  [B][npad*npad]  L (lower tiles, K = L L^T) and V = L^-T (strictly-upper tiles)
//   Dinv/DinvT [B][J][NB*NB]  inverse of each diagonal block of L, and its transpose
struct gprb_batch {
  gprb_ctx* ctx = nullptr;
  int32_t B = 0;
  int64_t n = 0, npad = 0;
  int32_t d = 0, J = 0, P = 0;
  int32_t kind = 0;
  std::vector<gprb_dataset*> ds;
  const double** Xptr = nullptr;   // device array [B] of dataset X pointers
  const double** Xtptr = nullptr;  // device array [B] of dataset Xt pointers
  double* ymm = nullptr;          // [B][npad] (zero padded)
  double* theta = nullptr;        // [B][P] theta of the last evaluation
  double* A = nullptr;
  double* Lm = nullptr;
  double* Dinv = nullptr;
  double* DinvT = nullptr;
  double* KinvD = nullptr;        // [B][J][NB*NB] diagonal tiles of K^-1
  double* alpha = nullptr;        // [B][npad]
  double* zbuf = nullptr;         // [B][npad] forward-substitution result
  double* jitter = nullptr;       // [B] diag_off + cumulative diagonal jitter added this evaluation
  double* diag_off = nullptr;     // [B] fixed per-GP diagonal offset (gprb_batch_set_diag_offset), default 0
  double* logdet_part = nullptr;  // [B][J]
  int32_t* fail = nullptr;        // [B] 0 ok / first failing column+1 (LAPACK info)
  double* mll = nullptr;          // [B]
  double* grad = nullptr;         // [B][P]
  double* grad_part = nullptr;    // [B][ntiles][P+1] per-tile partial sums (deterministic 2-pass reduction)
  int32_t* list = nullptr;        // [2B] compact lists of GP indices: [0,B) the stream groups of a pass, [B,2B) the fresh / retried GPs
  int32_t* list_host = nullptr;   // pinned, same layout
  std::vector<int32_t> tries;     // per GP: make_posdef! jitter additions of the evaluation in progress
  int32_t* fail_host = nullptr;   // pinned
  double* stage_host = nullptr;   // pinned staging for theta / results
  int64_t stage_doubles = 0;
  cudaStream_t stream[gprb::MAX_STREAMS] = {};
  int nstreams = 1;
  int rl_max = 24;                // passes with at most this many GPs use the right-looking (low-latency) factorisation
  double group_skew = 0.0;        // stream groups of a pass get sizes proportional to 1 + skew .. 1 - skew (GPRB200_GROUP_SKEW)
  int solve_cluster_below = 0;    // passes with fewer GPs than this use k_solve_cluster (GPRB200_SOLVE_CLUSTER_BELOW, default SM count)
  cudaEvent_t ev[8] = {};
  cudaEvent_t join[gprb::MAX_STREAMS] = {};
  bool profiling = false;
  std::vector<uint8_t> state_ok;  // per GP: factor + alpha resident (last evaluation succeeded)
  std::vector<uint8_t> inv_ok;    // per GP: K^-1 resident in A (last evaluation was value+gradient)
  std::vector<uint8_t> v_ok;      // per GP: V = L^-T resident in the upper tiles of Lm (TRTRI stage done)
  // state reuse (api.cu:eval_pass): theta / info / dataset version of the last successful host-theta evaluation per GP
  std::vector<double> theta_last;
  std::vector<uint8_t> theta_valid;
  std::vector<int32_t> info_last;
  std::vector<uint64_t> ds_ver;
  double stage_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  // prediction pipelines (scratch allocated on first use and kept, grow-only): slot s runs on stream[4s .. 4s+3]
  gprb_predict_slot ps[2];
  gprb_postcov_ws pc;             // full covariance / posterior draws (gprb_predict_cov, gprb_sample_posterior)
  gprb_loo_ws loo;                // leave-one-out cross-validation (gprb_eval_loo)
  gprb_predgrad_ws pg;            // predictive gradients (gprb_predict_grad)
  // The tile GEMM's arguments on the batch's factor, which every tile-GEMM launch on it starts from: Lm, A (Cin), Dinv,
  // DinvT, KinvD, fail, their strides and the TMA tensor maps of the operands, encoded once per batch (box = padded rows
  // x KT columns x 1 GP; tm_LT: Lm with box = KT rows x 128 columns, GEMM_BWD_ROW reads L's lower tiles transposed)
  gprb::GemmArgs gemm{};
  std::vector<cudaEvent_t> gemm_ev;  // profiling: start/stop pairs around every tile-GEMM launch
  int gemm_ev_used = 0;
  std::vector<double> gemm_ms;  // per tile-GEMM launch time of the last profiled evaluation, launch order
};

// --------------------------------------------------------------------------------------
// device-side PTX helpers (sm_100a): mbarrier, bulk async copy (TMA engine, SASS UBLKCP), DMMA
// --------------------------------------------------------------------------------------
#ifdef __CUDACC__
namespace gprb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// 1-D bulk copy global -> shared through the TMA engine; completion counted in bytes on `bar`.
// dst, src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// 3-D tiled TMA load (SASS UTMALDG): the box at element coordinates (c0 = row, c1 = column, c2 = GP) of the tensor map
// lands densely at dst (128-byte aligned); completion is counted in bytes on `bar` (always the full box, out-of-range
// elements arrive as zeros).
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
                   smem_u32(dst)),
               "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
               : "memory");
}
// The same box, fetched into L2 only (SASS UTMAPF): no shared memory, no barrier, no register - a hint for a later load.
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* map, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(map), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// Order generic-proxy smem writes before later async-proxy (TMA) accesses to the same smem.
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// exp(x) for x <= 0, branch-free (the library exp carries range-check branches that keep the compiler from
// interleaving neighbouring evaluations; the pairwise kernels evaluate 64 per thread).  Cody-Waite reduction with
// k = rint(x log2 e), degree-13 Taylor polynomial on |r| <= ln2/2 (truncation 4e-18), 2^k applied as two exact
// power-of-two factors so gradual underflow needs no special case.  <= 1 ulp in the normal range (tests/test_oracle
// pins it against numpy through the K parity bound); x < -800 is clamped (exp underflows to 0), NaN propagates.
__device__ __forceinline__ double exp_nonpos(double x) {
  const double xc = x < -800.0 ? -800.0 : x;
  const double t = fma(xc, 1.4426950408889634, 6755399441055744.0);
  const double k = t - 6755399441055744.0;
  const int ki = __double2loint(t);
  double r = fma(k, -6.93147180369123816490e-01, xc);
  r = fma(k, -1.90821492927058770002e-10, r);
  double p = 1.6059043836821613e-10;        // 1/13!
  p = fma(p, r, 2.08767569878681e-09);      // 1/12!
  p = fma(p, r, 2.505210838544172e-08);     // 1/11!
  p = fma(p, r, 2.755731922398589e-07);     // 1/10!
  p = fma(p, r, 2.7557319223985893e-06);    // 1/9!
  p = fma(p, r, 2.48015873015873e-05);      // 1/8!
  p = fma(p, r, 1.984126984126984e-04);     // 1/7!
  p = fma(p, r, 1.388888888888889e-03);     // 1/6!
  p = fma(p, r, 8.333333333333333e-03);     // 1/5!
  p = fma(p, r, 4.1666666666666664e-02);    // 1/4!
  p = fma(p, r, 1.6666666666666666e-01);    // 1/3!
  p = fma(p, r, 0.5);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  const int k1 = ki >> 1, k2 = ki - k1;
  return p * __hiloint2double((k1 + 1023) << 20, 0) * __hiloint2double((k2 + 1023) << 20, 0);
}

// k(r2) of the kernel family KIND for the weighted squared distance r2 (predict.cu, postcov.cu)
template <int KIND>
__device__ __forceinline__ double kcross(double r2, double sf2) {
  if (KIND == GPRB_KERNEL_SE_ARD) return sf2 * exp_nonpos(-0.5 * r2);
  const double r = sqrt(r2);
  if (KIND == GPRB_KERNEL_MAT12_ARD) return sf2 * exp_nonpos(-r);
  if (KIND == GPRB_KERNEL_MAT32_ARD) { const double s = 1.7320508075688772 * r; return sf2 * (1.0 + s) * exp_nonpos(-s); }
  const double s = 2.23606797749979 * r;
  return sf2 * (1.0 + s + 5.0 * r2 / 3.0) * exp_nonpos(-s);
}

// D(8x8) += A(8x4, row) * B(4x8, col) in fp64 on the tensor pipe (SASS DMMA.8x8x4).
// lane = 4*g + t : a = A[g][t], b = B[t][g] (i.e. "B^T row g, col t"), c0/c1 = D[g][2t], D[g][2t+1].
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

}  // namespace gprb
#endif
