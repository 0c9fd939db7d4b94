// C ABI of libgprb200 (include/gprb200.h): handle management and the host-side orchestration of the
// evaluation pipeline  assembly -> blocked Cholesky -> solves/mll -> inverse -> fused gradient.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <limits>
#include <new>
#include <type_traits>
#include <unordered_set>

#include "common.cuh"
#include "kernels.h"

namespace gprb {

static thread_local std::string g_err = "";
void set_error(const std::string& msg) { g_err = msg; }
int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  g_err = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what + " (" + file + ":" + std::to_string(line) + ")";
  return e == cudaErrorMemoryAllocation ? GPRB_ERR_NOMEM : GPRB_ERR_CUDA;
}

// fresh evaluation: the diagonal term starts at the GP's fixed offset (gprb_batch_set_diag_offset, default 0)
__global__ void k_reset_jitter(double* jitter, const double* diag_off, const int32_t* list, int count) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < count) jitter[list[k]] = diag_off[list[k]];
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
int make_tensor_map(CUtensorMap* map, const double* base, uint64_t rows, uint64_t cols, uint64_t gps, uint64_t col_stride_doubles,
                    uint64_t gp_stride_doubles, uint32_t box_rows, uint32_t box_cols) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
      set_error("cuTensorMapEncodeTiled is not available from this driver (TMA tensor maps are required)");
      return GPRB_ERR_CUDA;
    }
    encode = reinterpret_cast<EncodeFn>(fn);
  }
  const cuuint64_t gdim[3] = {rows, cols, gps};
  const cuuint64_t gstride[2] = {col_stride_doubles * sizeof(double), gp_stride_doubles * sizeof(double)};
  const cuuint32_t box[3] = {box_rows, box_cols, 1};
  const cuuint32_t estride[3] = {1, 1, 1};
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<double*>(base), gdim, gstride, box, estride,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    return GPRB_ERR_CUDA;
  }
  return 0;
}

// Operand tensor maps of the tile GEMM on B factors ga.Lm [B][npad][npad], beside ga.Cin (K) and the inverted diagonal
// blocks ga.Dinv / ga.DinvT [B][J*128][128]: padded boxes (132 / 68 rows) x KT columns x one GP
static int encode_factor_maps(GemmArgs& ga, uint64_t B) {
  const uint64_t np = ga.npad, nd = (uint64_t)ga.J * NB, ms = ga.mat_stride, ds = ga.dinv_stride;
  int rc;
  if ((rc = make_tensor_map(&ga.tm_L132, ga.Lm, np, np, B, np, ms, NB + 4, KT)) ||
      (rc = make_tensor_map(&ga.tm_L68, ga.Lm, np, np, B, np, ms, NB / 2 + 4, KT)) ||
      (rc = make_tensor_map(&ga.tm_A68, ga.Cin, np, np, B, np, ms, NB / 2 + 4, KT)) ||
      (rc = make_tensor_map(&ga.tm_DT132, ga.DinvT, NB, nd, B, NB, ds, NB + 4, KT)) ||
      (rc = make_tensor_map(&ga.tm_DT68, ga.DinvT, NB, nd, B, NB, ds, NB / 2 + 4, KT)) ||
      (rc = make_tensor_map(&ga.tm_D132, ga.Dinv, NB, nd, B, NB, ds, NB + 4, KT)))
    return rc;
  return 0;
}

// The batch's tile-GEMM prototype (gprb_batch::gemm) on its current buffers, n and npad, tensor maps included.
static int set_batch_gemm(gprb_batch* b) {
  const int64_t mat = b->npad * b->npad, dinv = (int64_t)b->J * NB * NB;
  b->gemm = GemmArgs{b->Lm, b->DinvT, b->Dinv, b->A, b->Lm, b->KinvD, nullptr, mat, dinv, (int)b->npad, b->J, 0, GEMM_CHOL_DIAG,
                     (int)((b->n + KT - 1) / KT * KT)};
  b->gemm.fail = b->fail;
  int rc;
  if ((rc = encode_factor_maps(b->gemm, (uint64_t)b->B)) ||
      (rc = make_tensor_map(&b->gemm.tm_LT, b->Lm, (uint64_t)b->npad, (uint64_t)b->npad, (uint64_t)b->B, (uint64_t)b->npad,
                            (uint64_t)mat, KT, NB)))
    return rc;
  return 0;
}

// make_posdef! after one factorisation attempt with status f (LAPACK info; < 0: no state or non-finite input): either one
// more jitter is due (tries counts it, returns true) or info gets the final outcome - the jitter count, -2, or -1 when
// the matrix is still indefinite after MAX_JITTER jitters.
static bool posdef_retry(int32_t f, int32_t& tries, int32_t& info) {
  if (f > 0 && tries < MAX_JITTER) { ++tries; return true; }
  info = f == 0 ? tries : f < 0 ? -2 : -1;
  return false;
}

template <typename T>
static int dev_alloc(T** p, size_t count) {
  *p = nullptr;
  if (count == 0) count = 1;
  cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
  if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc", __FILE__, __LINE__);
  return 0;
}

// The datasets of a batch, each once, in order of first use by GP index.
static std::vector<gprb_dataset*> distinct_datasets(const gprb_batch* b) {
  std::vector<gprb_dataset*> out;
  std::unordered_set<gprb_dataset*> seen;
  for (gprb_dataset* d : b->ds)
    if (seen.insert(d).second) out.push_back(d);
  return out;
}

static void free_batch(gprb_batch* b) {
  if (!b) return;
  cudaFree(b->Xptr); cudaFree(b->Xtptr); cudaFree(b->ymm); cudaFree(b->theta); cudaFree(b->A); cudaFree(b->Lm);
  cudaFree(b->Dinv); cudaFree(b->DinvT); cudaFree(b->KinvD); cudaFree(b->alpha); cudaFree(b->zbuf); cudaFree(b->jitter); cudaFree(b->diag_off);
  cudaFree(b->logdet_part); cudaFree(b->fail); cudaFree(b->mll); cudaFree(b->grad);
  cudaFree(b->grad_part); cudaFree(b->list);
  for (gprb_predict_slot& sl : b->ps) {
    cudaFree(sl.pX); cudaFree(sl.pms); cudaFree(sl.pmu); cudaFree(sl.pvar); cudaFree(sl.pT); cudaFree(sl.pmupart);
    cudaFree(sl.pq); cudaFree(sl.pcount); cudaFree(sl.mask);
    if (sl.h_in) cudaFreeHost(sl.h_in);
    if (sl.h_out) cudaFreeHost(sl.h_out);
    if (sl.h_mask) cudaFreeHost(sl.h_mask);
    if (sl.t0) cudaEventDestroy(sl.t0);
    if (sl.t1) cudaEventDestroy(sl.t1);
  }
  {
    gprb_postcov_ws& w = b->pc;
    cudaFree(w.T); cudaFree(w.S); cudaFree(w.L); cudaFree(w.Dinv); cudaFree(w.DinvT); cudaFree(w.logdet); cudaFree(w.Z);
    cudaFree(w.O); cudaFree(w.bad); cudaFree(w.fail); cudaFree(w.list);
    if (w.fail_host) cudaFreeHost(w.fail_host);
    if (w.list_host) cudaFreeHost(w.list_host);
    if (w.z_ready) cudaEventDestroy(w.z_ready);
  }
  {
    gprb_loo_ws& w = b->loo;
    cudaFree(w.M); cudaFree(w.W); cudaFree(w.KD); cudaFree(w.vec); cudaFree(w.part); cudaFree(w.mll); cudaFree(w.out); cudaFree(w.skip);
    if (w.skip_host) cudaFreeHost(w.skip_host);
  }
  cudaFree(b->pg.jac); cudaFree(b->pg.dms);
  if (b->list_host) cudaFreeHost(b->list_host);
  if (b->fail_host) cudaFreeHost(b->fail_host);
  if (b->stage_host) cudaFreeHost(b->stage_host);
  for (int s = 0; s < MAX_STREAMS; ++s) {
    if (b->stream[s]) cudaStreamDestroy(b->stream[s]);
    if (b->join[s]) cudaEventDestroy(b->join[s]);
  }
  for (int s = 0; s < 8; ++s)
    if (b->ev[s]) cudaEventDestroy(b->ev[s]);
  for (cudaEvent_t e : b->gemm_ev) cudaEventDestroy(e);
  delete b;
}

// Enqueue one evaluation of the GPs in list[off .. off+count) on `st`: inverse + fused gradient for the first `ngrad`
// entries of the segment (the host orders value+gradient GPs first); assembly, Cholesky and solve for all entries but
// the first `nreuse` (<= ngrad), whose factor, alpha and mll of the previous evaluation at the same theta are still
// resident (the optimiser asks for the gradient at the point its line search just accepted).
// `ops` != nullptr: the launches are not issued but appended (as closures) to `ops`, so that run_pipeline can issue the
// launches of all stream groups interleaved - every group then starts at once instead of one enqueue time (0.3 ms of host
// work per group) after the previous one, which matters for short passes (50 GPs per GPU in the 8-GPU strong split).
// j0 > 0 (gprb_batch_append, left-looking, value only): the block rows < j0 of K, L, Dinv and the logdet partials are
// resident and final - only the lower tiles in block rows >= j0 are assembled, block columns j < j0 get their CHOL_COL
// tiles in those rows, block columns >= j0 the whole left-looking step, and the solve runs over the whole factor.
using LaunchOps = std::vector<std::function<int()>>;
static int enqueue_pipeline(gprb_batch* b, int off, int count, int ngrad, int nreuse, bool right_looking, cudaStream_t st,
                            bool prof, LaunchOps* ops = nullptr, int j0 = 0) {
  if (count <= 0) return 0;
  const bool with_grad = ngrad > 0;
  const int32_t* glist = b->list + off;     // inverse + gradient: glist[0 .. ngrad)
  const int32_t* list = glist + nreuse;     // assembly, factorisation, solves: list[0 .. count)
  count -= nreuse;
  const int J = b->J;
  const int64_t ms = b->npad * b->npad, dstride = (int64_t)J * NB * NB;
  int rc;
  int64_t& launches = b->ctx->launches;
  int gcount = count;  // GPs per tile-GEMM launch (count for the factorisation, ngrad for the inverse)
  auto run = [&](std::function<int()> f) -> int {
    if (ops) { ops->push_back(std::move(f)); return 0; }
    return f();
  };
  auto gemm = [&](const GemmArgs& a, int ntiles) -> int {
    const int count = gcount;
    if (!prof) return run([a, ntiles, count, st] { return launch_tile_gemm(a, ntiles, count, st); });
    while ((int)b->gemm_ev.size() < b->gemm_ev_used + 2) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) return cuda_fail(cudaGetLastError(), "cudaEventCreate", __FILE__, __LINE__);
      b->gemm_ev.push_back(e);
    }
    cudaEventRecord(b->gemm_ev[b->gemm_ev_used], st);
#ifdef GPRB_TIMELINE
    // debug build only: per-tile phase timestamps of this launch, averaged and printed to stderr
    static unsigned long long* tl_dev = nullptr;
    const size_t tl_n = (size_t)count * ntiles * 2 * 8;  // two half-tile CTAs per logical tile (FWD_ROW: one; the rest stays zero)
    if (!tl_dev) cudaMalloc(&tl_dev, sizeof(unsigned long long) * 8 * 65536 * 16);
    cudaMemsetAsync(tl_dev, 0, sizeof(unsigned long long) * tl_n, st);
    GemmArgs a2 = a; a2.tl = tl_dev;
    int r = launch_tile_gemm(a2, ntiles, count, st);
    cudaEventRecord(b->gemm_ev[b->gemm_ev_used + 1], st);
    b->gemm_ev_used += 2;
    {
      std::vector<unsigned long long> h(tl_n);
      cudaStreamSynchronize(st);
      cudaMemcpy(h.data(), tl_dev, sizeof(unsigned long long) * tl_n, cudaMemcpyDeviceToHost);
      double ph[6] = {0, 0, 0, 0, 0, 0}, tot = 0, waitc = 0; size_t cnt = 0;
      for (size_t k = 0; k < tl_n; k += 8) {
        const unsigned long long* t = &h[k];
        if (!t[0] || !t[6]) continue;
        unsigned long long prev = t[0];
        for (int q = 1; q <= 6; ++q) { unsigned long long cur = t[q] ? t[q] : prev; ph[q - 1] += (double)(cur - prev); prev = cur; }
        tot += (double)(t[6] - t[0]); waitc += (double)t[7]; ++cnt;
      }
      if (cnt) fprintf(stderr, "TL mode %d step %2d tiles %6zu  fill %6.2f main %7.2f cin %6.2f park %6.2f post %6.2f store %6.2f  total %7.2f us  (operand wait in main, after the first chunk %6.2f us)\n",
                       a.mode, a.step, cnt, ph[0] / cnt / 1e3, ph[1] / cnt / 1e3, ph[2] / cnt / 1e3, ph[3] / cnt / 1e3, ph[4] / cnt / 1e3, ph[5] / cnt / 1e3, tot / cnt / 1e3, waitc / cnt / 1965.0);
    }
    return r;
#else
    int r = launch_tile_gemm(a, ntiles, count, st);
    cudaEventRecord(b->gemm_ev[b->gemm_ev_used + 1], st);
    b->gemm_ev_used += 2;
    return r;
#endif
  };
  if (prof) { b->gemm_ev_used = 0; cudaEventRecord(b->ev[0], st); }
  const int nv = (int)((b->n + KT - 1) / KT * KT);
  GemmArgs ga = b->gemm;
  ga.list = list;
  { static const int pf = getenv("GPRB200_PF_CIN") ? atoi(getenv("GPRB200_PF_CIN")) : 1; ga.pf_cin = (!right_looking && pf) ? 1 : 0; }
  if (count > 0) {
  // Small passes are latency bound (one dependent chain of 3 J launches): they use the right-looking factorisation,
  // whose launches are short and wide, instead of the left-looking one, whose k-loops grow with the column index.
  AssembleArgs aa{b->Xtptr, b->theta, b->jitter, b->A, nullptr, b->fail, list, ms, (int)b->n, (int)b->npad, b->d, J, b->kind};
  aa.tile0 = j0 * (j0 + 1) / 2;
  if (right_looking) aa.A2 = b->Lm;
  if ((rc = run([aa, count, st] { return launch_assemble(aa, count, st); }))) return rc;
  ++launches;
  if (prof) cudaEventRecord(b->ev[1], st);
  DiagArgs da{nullptr, b->Lm, b->Dinv, b->DinvT, b->logdet_part, b->fail, list, ms, dstride, (int)b->npad, J, 0, nv};
  if (right_looking) ga.Cin = b->Lm;  // S lives (and is updated in place) in the lower tiles of Lm
  for (int j = 0; j < J; ++j) {
    ga.step = j;
    if (j < j0) {
      ga.mode = GEMM_CHOL_COL; ga.row0 = j0;
      if ((rc = gemm(ga, J - j0))) return rc;
      ++launches;
      ga.row0 = 0;
      continue;
    }
    if (!right_looking && j > 0) {  // S(0,0) = K(0,0): k_diag_factor reads block column 0 straight from A
      ga.mode = GEMM_CHOL_DIAG;
      if ((rc = gemm(ga, 1))) return rc;
      ++launches;
    }
    da.step = j;
    da.Src = (!right_looking && j == 0) ? b->A : nullptr;
    if ((rc = run([da, count, st] { return launch_diag_factor(da, count, st); }))) return rc;
    ++launches;
    if (j + 1 < J) {
      ga.mode = right_looking ? GEMM_CHOL_PANEL : GEMM_CHOL_COL;
      if ((rc = gemm(ga, J - 1 - j))) return rc;
      ++launches;
      if (right_looking) {
        ga.mode = GEMM_CHOL_TRAIL;
        if ((rc = gemm(ga, (J - 1 - j) * (J - j) / 2))) return rc;
        ++launches;
      }
    }
  }
  if (prof) cudaEventRecord(b->ev[2], st);
  SolveArgs sa{b->Lm, b->Dinv, b->ymm, b->logdet_part, b->fail, b->zbuf, b->alpha, b->mll, list, ms, dstride,
               (int)b->n, (int)b->npad, J, nv};
  sa.cluster_below = b->solve_cluster_below;
  if ((rc = run([sa, count, st] { return launch_solve(sa, count, st); }))) return rc;
  ++launches;
  }
  if (prof) cudaEventRecord(b->ev[3], st);
  if (with_grad) {
    ga.Cin = nullptr;
    ga.list = glist;
    gcount = ngrad;
    for (int i = 1; i < J; ++i) {
      ga.step = i; ga.mode = GEMM_TRTRI_ROW; ga.Cout = b->Lm;
      if ((rc = gemm(ga, i))) return rc;
      ++launches;
    }
    ga.mode = GEMM_LAUUM; ga.step = 0; ga.Cout = b->A;
    if ((rc = gemm(ga, J * (J + 1) / 2))) return rc;
    ++launches;
    if (prof) cudaEventRecord(b->ev[4], st);
    GradArgs gr{b->Xtptr, b->theta, b->A, b->KinvD, b->alpha, b->grad_part, b->grad, b->fail, glist, ms, dstride,
                (int)b->n, (int)b->npad, b->d, J, b->kind};
    if ((rc = run([gr, ngrad, st] { return launch_grad(gr, ngrad, st); }))) return rc;
    launches += 2;
    if (prof) cudaEventRecord(b->ev[5], st);
  }
  return 0;
}

// One stream group of an evaluation pass: list[off .. off+count), the first ngrad of them with gradient, the first
// nreuse of those on the resident factorisation.
struct Group { int off, count, ngrad, nreuse; bool rl; int j0 = 0; };

// Order the active GPs of a pass into stream groups inside list_host: the value+gradient GPs and the value-only GPs
// are each dealt evenly over the groups (equal work per stream), gradient GPs first inside every group.
static std::vector<Group> build_groups(gprb_batch* b, const std::vector<int32_t>& reuse_gps, const std::vector<int32_t>& grad_gps,
                                       const std::vector<int32_t>& val_gps) {
  const int total = (int)(reuse_gps.size() + grad_gps.size() + val_gps.size());
  const int S = (b->profiling || total < 8 || total <= b->rl_max || b->nstreams == 1) ? 1 : b->nstreams;
  std::vector<Group> groups;
  int off = 0;
  // Unequal group sizes (weights 1 + skew, ..., 1 - skew): equal groups start together and run the same launches, so
  // they reach their low-occupancy phases (diagonal tiles, potf2, the first rows of the triangular inverse) at the same
  // time; groups of different size drift apart, and the thin phases of one fall under the wide phases of another.
  std::vector<double> cum(S + 1, 0.0);
  for (int s = 0; s < S; ++s) cum[s + 1] = cum[s] + (S > 1 ? 1.0 + b->group_skew * (double)(S - 1 - 2 * s) / (double)(S - 1) : 1.0);
  auto cut = [&](size_t m, int s) { return (int)llround((double)m * cum[s] / cum[S]); };
  for (int s = 0; s < S; ++s) {
    const int r0 = cut(reuse_gps.size(), s), r1 = cut(reuse_gps.size(), s + 1);
    const int g0 = cut(grad_gps.size(), s), g1 = cut(grad_gps.size(), s + 1);
    const int v0 = cut(val_gps.size(), s), v1 = cut(val_gps.size(), s + 1);
    Group g{off, (r1 - r0) + (g1 - g0) + (v1 - v0), (r1 - r0) + (g1 - g0), r1 - r0, !b->profiling && total <= b->rl_max, 0};
    for (int k = r0; k < r1; ++k) b->list_host[off++] = reuse_gps[k];
    for (int k = g0; k < g1; ++k) b->list_host[off++] = grad_gps[k];
    for (int k = v0; k < v1; ++k) b->list_host[off++] = val_gps[k];
    if (g.count > 0) groups.push_back(g);
  }
  return groups;
}

// Run one pass: every group on its own stream so the serial diagonal-block kernels of one group overlap the DMMA
// tiles of another.  Joins everything on stream[0].
static int run_pipeline(gprb_batch* b, const std::vector<Group>& groups) {
  int rc;
  if (groups.empty()) return 0;
  if (b->profiling) {
    const Group& g = groups[0];
    if ((rc = enqueue_pipeline(b, g.off, g.count, g.ngrad, g.nreuse, g.rl, b->stream[0], true, nullptr, g.j0))) return rc;
    GPRB_CUDA(cudaStreamSynchronize(b->stream[0]));
    float ms = 0.f;
    const int last = g.ngrad > 0 ? 5 : 3;
    for (int s = 0; s < 5; ++s) b->stage_ms[s] = 0.0;
    for (int s = 0; s < last; ++s) {
      GPRB_CUDA(cudaEventElapsedTime(&ms, b->ev[s], b->ev[s + 1]));
      b->stage_ms[s] = ms;
    }
    GPRB_CUDA(cudaEventElapsedTime(&ms, b->ev[0], b->ev[last]));
    b->stage_ms[5] = ms;
    double gsum = 0.0;
    b->gemm_ms.clear();
    for (int k = 0; k + 1 < b->gemm_ev_used; k += 2) {
      GPRB_CUDA(cudaEventElapsedTime(&ms, b->gemm_ev[k], b->gemm_ev[k + 1]));
      gsum += ms;
      b->gemm_ms.push_back(ms);
    }
    b->stage_ms[6] = gsum;
    b->stage_ms[7] = b->gemm_ev_used / 2;
    return 0;
  }
  GPRB_CUDA(cudaEventRecord(b->join[0], b->stream[0]));
  std::vector<LaunchOps> ops(groups.size());
  size_t longest = 0;
  for (size_t s = 0; s < groups.size(); ++s) {
    const Group& g = groups[s];
    if (s > 0) GPRB_CUDA(cudaStreamWaitEvent(b->stream[s], b->join[0], 0));
    if ((rc = enqueue_pipeline(b, g.off, g.count, g.ngrad, g.nreuse, g.rl, b->stream[s], false, groups.size() > 1 ? &ops[s] : nullptr,
                               g.j0)))
      return rc;
    longest = std::max(longest, ops[s].size());
  }
  for (size_t k = 0; k < longest; ++k)  // launch k of every group, group by group: all groups advance together
    for (size_t s = 0; s < groups.size(); ++s)
      if (k < ops[s].size() && (rc = ops[s][k]())) return rc;
  for (size_t s = 1; s < groups.size(); ++s) {
    GPRB_CUDA(cudaEventRecord(b->join[s], b->stream[s]));
    GPRB_CUDA(cudaStreamWaitEvent(b->stream[0], b->join[s], 0));
  }
  return 0;
}

// ONE pipeline pass over the GPs with mode != 0 (theta already on the device).  retry[gp] != 0: the GP's previous
// pass failed its factorisation - its cumulative jitter grows by 1e-6 tr(K)/n (make_posdef!) instead of being reset.
// Afterwards: info[gp] final for the GPs that are done, pending[gp] = 1 for those that need another retry pass.
//
// State reuse (theta_host != nullptr): a GP asked to evaluate, first try, at exactly the theta of its last successful
// evaluation (same dataset upload) keeps what is resident - a value-only request is answered from the resident mll, a
// gradient request only runs the inverse and the fused gradient on the resident factor (or nothing, when that gradient
// is resident too).  The results are bit-identical to a fresh evaluation: every stage is deterministic, and the jitter
// the earlier evaluation settled on is the one make_posdef! would arrive at again.  This is the optimiser's pattern:
// the reference evaluates the point a line search accepts twice (value, then value + gradient), and once more after
// the last iteration.
static int eval_pass(gprb_batch* b, const double* theta_host, const uint8_t* mode, const uint8_t* retry,
                     std::vector<int32_t>& info, std::vector<uint8_t>& pending) {
  int rc;
  const int B = b->B, P = b->P;
  if ((int)b->tries.size() != B) b->tries.assign(B, 0);
  if ((int)b->theta_valid.size() != B) {
    b->theta_valid.assign(B, 0); b->theta_last.assign((size_t)B * P, 0.0); b->info_last.assign(B, 0); b->ds_ver.assign(B, 0);
  }
  pending.assign(B, 0);
  static const bool allow_reuse = [] { const char* e = getenv("GPRB200_REUSE"); return !(e && e[0] == '0'); }();
  std::vector<int32_t> reuse_gps, grad_gps, val_gps, cached;
  int nfresh = 0, nretry = 0;
  int32_t* aux = b->list_host + B;  // fresh GPs from the front, retried GPs from the back
  for (int i = 0; i < B; ++i) {
    if (!mode[i]) continue;
    const bool is_retry = retry && retry[i];
    if (allow_reuse && theta_host && !is_retry && !b->profiling && b->state_ok[i] && b->theta_valid[i] &&
        b->ds_ver[i] == b->ds[i]->version &&
        memcmp(theta_host + (size_t)i * P, b->theta_last.data() + (size_t)i * P, sizeof(double) * P) == 0) {
      if (mode[i] == 1 || b->inv_ok[i]) cached.push_back(i);  // everything asked for is resident
      else reuse_gps.push_back(i);                             // gradient on the resident factor
      continue;
    }
    (mode[i] == 2 ? grad_gps : val_gps).push_back(i);
    if (is_retry) aux[B - 1 - nretry++] = i;
    else { aux[nfresh++] = i; b->tries[i] = 0; }
  }
  for (int gp : cached) info[gp] = b->info_last[gp];
  const int count = (int)(reuse_gps.size() + grad_gps.size() + val_gps.size());
  if (count == 0) return 0;
  const std::vector<Group> groups = build_groups(b, reuse_gps, grad_gps, val_gps);
  GPRB_CUDA(cudaMemcpyAsync(b->list, b->list_host, sizeof(int32_t) * 2 * B, cudaMemcpyHostToDevice, b->stream[0]));
  if (nfresh) {
    k_reset_jitter<<<(nfresh + 127) / 128, 128, 0, b->stream[0]>>>(b->jitter, b->diag_off, b->list + B, nfresh);
    GPRB_CUDA(cudaGetLastError());
  }
  if (nretry && (rc = launch_add_jitter(b->theta, b->jitter, b->list + 2 * B - nretry, b->d, nretry, b->stream[0]))) return rc;
  if ((rc = run_pipeline(b, groups))) return rc;
  GPRB_CUDA(cudaMemcpyAsync(b->fail_host, b->fail, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, b->stream[0]));
  GPRB_CUDA(cudaStreamSynchronize(b->stream[0]));
  if (getenv("GPRB200_LBFGS_TRACE")) {  // where do failed factorisations break down? (first bad pivot / n)
    double sum = 0; int nf = 0;
    for (int gp = 0; gp < B; ++gp)
      if (mode[gp] && b->fail_host[gp] > 0) { sum += (double)b->fail_host[gp] / (double)b->n; ++nf; }
    if (nf) fprintf(stderr, "  pass: %d of %d factorisations failed, mean failing pivot at %.2f n\n", nf, count, sum / nf);
  }
  for (int gp : reuse_gps) { info[gp] = b->info_last[gp]; b->inv_ok[gp] = 1; b->v_ok[gp] = 1; }
  for (int pass = 0; pass < 2; ++pass)
    for (int gp : (pass == 0 ? grad_gps : val_gps)) {
      b->theta_valid[gp] = 0;
      if (posdef_retry(b->fail_host[gp], b->tries[gp], info[gp])) {
        pending[gp] = 1; b->state_ok[gp] = 0; b->inv_ok[gp] = 0; b->v_ok[gp] = 0;
        continue;
      }
      b->state_ok[gp] = info[gp] >= 0;
      b->inv_ok[gp] = pass == 0 && info[gp] >= 0;
      b->v_ok[gp] = b->inv_ok[gp];
      if (info[gp] >= 0) b->info_last[gp] = info[gp];  // the jitter rung of the resident state (gprb_batch_append reads it)
      if (theta_host && info[gp] >= 0) {  // remember what is resident now
        memcpy(b->theta_last.data() + (size_t)gp * P, theta_host + (size_t)gp * P, sizeof(double) * P);
        b->theta_valid[gp] = 1;
        b->ds_ver[gp] = b->ds[gp]->version;
      }
    }
  return 0;
}

// Evaluation with the make_posdef! retry loop inside (gprb_eval / gprb_eval_mixed / gprb_eval_device): passes are
// repeated for the GPs that still need a jitter until none is pending.
static int evaluate_modes(gprb_batch* b, const double* theta_host, const uint8_t* mode, std::vector<int32_t>& info) {
  info.assign(b->B, 0);
  std::vector<uint8_t> cur(mode, mode + b->B), retry(b->B, 0), pending;
  for (;;) {
    int rc = eval_pass(b, theta_host, cur.data(), retry.data(), info, pending);
    if (rc) return rc;
    bool any = false;
    for (int i = 0; i < b->B; ++i) {
      cur[i] = pending[i] ? cur[i] : 0;
      retry[i] = pending[i];
      any = any || pending[i];
    }
    if (!any) return 0;
  }
}

// theta rows of the listed GPs -> device (pinned staging, one strided copy per contiguous run of GP indices)
static int upload_theta_rows(gprb_batch* b, const double* theta, const std::vector<int32_t>& act) {
  const int P = b->P, count = (int)act.size();
  double* st = b->stage_host;
  for (int k = 0; k < count; ++k) memcpy(st + (size_t)k * P, theta + (size_t)act[k] * P, sizeof(double) * P);
  for (int k = 0; k < count;) {
    int k2 = k + 1;
    while (k2 < count && act[k2] == act[k2 - 1] + 1) ++k2;
    GPRB_CUDA(cudaMemcpyAsync(b->theta + (size_t)act[k] * P, st + (size_t)k * P, sizeof(double) * P * (k2 - k),
                              cudaMemcpyHostToDevice, b->stream[0]));
    k = k2;
  }
  return 0;
}

// mll (+ grad rows of the mode-2 GPs) of the finished GPs -> host arrays
static int download_results(gprb_batch* b, const uint8_t* mode, const std::vector<int32_t>& info, const uint8_t* skip,
                            double* mll, double* grad, int32_t* info_out) {
  const int B = b->B, P = b->P;
  bool any_grad = false;
  for (int i = 0; i < B; ++i) any_grad = any_grad || (mode[i] == 2 && !(skip && skip[i]));
  double* res = b->stage_host;  // [B] mll then [B*P] grad
  GPRB_CUDA(cudaMemcpyAsync(res, b->mll, sizeof(double) * B, cudaMemcpyDeviceToHost, b->stream[0]));
  if (any_grad) GPRB_CUDA(cudaMemcpyAsync(res + B, b->grad, sizeof(double) * B * P, cudaMemcpyDeviceToHost, b->stream[0]));
  GPRB_CUDA(cudaStreamSynchronize(b->stream[0]));
  const double ninf = -std::numeric_limits<double>::infinity(), qnan = std::numeric_limits<double>::quiet_NaN();
  for (int gp = 0; gp < B; ++gp) {
    if (!mode[gp] || (skip && skip[gp])) continue;
    info_out[gp] = info[gp];
    const bool ok = info[gp] >= 0;
    mll[gp] = ok ? res[gp] : ninf;
    if (mode[gp] == 2)
      for (int p = 0; p < P; ++p) grad[(size_t)gp * P + p] = ok ? res[B + (size_t)gp * P + p] : qnan;
  }
  return 0;
}

int eval_pass_host(gprb_batch* b, const double* theta, const uint8_t* mode, const uint8_t* retry, double* mll, double* grad,
                   int32_t* info_out, uint8_t* pending_out) {
  GPRB_REQUIRE(b && theta && mode && mll && grad && info_out && pending_out, "eval_pass_host: NULL argument");
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  std::vector<int32_t> fresh;
  for (int i = 0; i < b->B; ++i)
    if (mode[i] && !(retry && retry[i])) fresh.push_back(i);
  int rc = upload_theta_rows(b, theta, fresh);
  if (rc) return rc;
  std::vector<int32_t> info(b->B, 0);
  std::vector<uint8_t> pending;
  if ((rc = eval_pass(b, theta, mode, retry, info, pending))) return rc;
  memcpy(pending_out, pending.data(), b->B);
  return download_results(b, mode, info, pending_out, mll, grad, info_out);
}

}  // namespace gprb

using namespace gprb;

extern "C" {

int gprb_version(void) { return 303; }
const char* gprb_last_error(void) { return g_err.c_str(); }

int gprb_init(gprb_ctx** out, int device) {
  GPRB_REQUIRE(out != nullptr, "gprb_init: ctx out-pointer is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error("gprb_init: no CUDA device visible - libgprb200 has no CPU fallback");
    return GPRB_ERR_NODEVICE;
  }
  GPRB_REQUIRE(device >= 0 && device < ndev, "gprb_init: device index out of range");
  cudaDeviceProp prop;
  GPRB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error(std::string("gprb_init: device '") + prop.name + "' is not sm_100 (B200); the library is built for sm_100a only");
    return GPRB_ERR_NODEVICE;
  }
  GPRB_CUDA(cudaSetDevice(device));
  // dynamic shared-memory opt-ins are per-device function attributes: set them for THIS device (a second context on
  // another GPU of the same process gets its own)
  int rc;
  if ((rc = configure_tile_gemm()) || (rc = configure_diag_factor()) || (rc = configure_post_cov())) return rc;
  gprb_ctx* c = new (std::nothrow) gprb_ctx();
  GPRB_REQUIRE(c != nullptr, "gprb_init: out of host memory");
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  int khz = 0;
  cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device);
  c->clock_khz = khz;
  c->l2_bytes = prop.l2CacheSize;
  cudaError_t se = cudaStreamCreateWithFlags(&c->upload, cudaStreamNonBlocking);
  if (se == cudaSuccess) se = cudaStreamCreateWithFlags(&c->upload2, cudaStreamNonBlocking);
  if (se == cudaSuccess) se = cudaEventCreateWithFlags(&c->upload_ev, cudaEventDisableTiming);
  if (se != cudaSuccess) { delete c; return cuda_fail(se, "cudaStreamCreate(upload)", __FILE__, __LINE__); }
  *out = c;
  return GPRB_OK;
}

int gprb_destroy(gprb_ctx* ctx) {
  if (ctx) {
    cudaSetDevice(ctx->device);
    comm_release(ctx);
    if (ctx->upload) cudaStreamDestroy(ctx->upload);
    if (ctx->upload2) cudaStreamDestroy(ctx->upload2);
    if (ctx->upload_ev) cudaEventDestroy(ctx->upload_ev);
  }
  delete ctx;
  return GPRB_OK;
}

int gprb_device_info(gprb_ctx* ctx, int64_t out[4]) {
  GPRB_REQUIRE(ctx && out, "gprb_device_info: NULL argument");
  GPRB_CUDA(cudaSetDevice(ctx->device));
  size_t fr = 0, tot = 0;
  GPRB_CUDA(cudaMemGetInfo(&fr, &tot));
  out[0] = ctx->sm_count; out[1] = ctx->clock_khz; out[2] = ctx->l2_bytes; out[3] = (int64_t)fr;
  return GPRB_OK;
}

int64_t gprb_launch_count(gprb_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ------------------------------------------------------------------------------------------------
// Enqueue the host -> device copy of one dataset on `st` (no synchronisation).
static int dataset_copy_async(gprb_dataset* ds, const double* X, int64_t ldx, cudaStream_t st) {
  ds->version++;  // evaluations on the previous contents are no longer reusable
  if (ldx == ds->d)
    GPRB_CUDA(cudaMemcpyAsync(ds->X, X, sizeof(double) * ds->d * ds->n, cudaMemcpyHostToDevice, st));
  else
    GPRB_CUDA(cudaMemcpy2DAsync(ds->X, sizeof(double) * ds->d, X, sizeof(double) * ldx, sizeof(double) * ds->d, ds->n,
                                cudaMemcpyHostToDevice, st));
  return 0;
}

// Enqueue the upload of one dataset (copy + transposed copy Xt) on the context's upload stream (no synchronisation).
static int dataset_upload_async(gprb_dataset* ds, const double* X, int64_t ldx) {
  cudaStream_t st = ds->ctx->upload;
  int rc = dataset_copy_async(ds, X, ldx, st);
  if (rc) return rc;
  if ((rc = launch_transpose_inputs(ds->X, ds->Xt, (int)ds->n, (int)ds->npad, ds->d, st))) return rc;
  ds->ctx->launches++;
  return 0;
}

static int dataset_upload(gprb_dataset* ds, const double* X, int64_t ldx) {
  GPRB_CUDA(cudaSetDevice(ds->ctx->device));
  int rc = dataset_upload_async(ds, X, ldx);
  if (rc) return rc;
  GPRB_CUDA(cudaStreamSynchronize(ds->ctx->upload));
  return 0;
}

int gprb_dataset_create(gprb_ctx* ctx, int64_t n, int32_t d, const double* X, int64_t ldx, gprb_dataset** out) {
  GPRB_REQUIRE(ctx && X && out, "gprb_dataset_create: NULL argument");
  *out = nullptr;
  GPRB_REQUIRE(n >= 1 && n <= (1 << 20), "gprb_dataset_create: n out of range");
  GPRB_REQUIRE(d >= 1 && d <= MAX_D, "gprb_dataset_create: d must be in 1..62");
  GPRB_REQUIRE(ldx >= d, "gprb_dataset_create: ldx < d");
  GPRB_CUDA(cudaSetDevice(ctx->device));
  gprb_dataset* ds = new (std::nothrow) gprb_dataset();
  GPRB_REQUIRE(ds != nullptr, "gprb_dataset_create: out of host memory");
  ds->ctx = ctx; ds->n = n; ds->d = d;
  ds->npad = (n + NB - 1) / NB * NB;
  int rc;
  if ((rc = dev_alloc(&ds->X, (size_t)n * d)) || (rc = dev_alloc(&ds->Xt, (size_t)ds->npad * d)) ||
      (rc = dataset_upload(ds, X, ldx))) {
    cudaFree(ds->X); cudaFree(ds->Xt); delete ds;
    return rc;
  }
  *out = ds;
  return GPRB_OK;
}

int gprb_dataset_update(gprb_dataset* ds, const double* X, int64_t ldx) {
  GPRB_REQUIRE(ds && X, "gprb_dataset_update: NULL argument");
  GPRB_REQUIRE(ldx >= ds->d, "gprb_dataset_update: ldx < d");
  return dataset_upload(ds, X, ldx);
}

// ds[0 .. count) are the members 0 .. count-1 of one slab, in order, and the host matrices form one contiguous block:
// the whole upload is ONE host->device copy and ONE transpose launch (the per-dataset form costs the host ~10 us per
// copy / launch to enqueue - 1 ms per 100 trial datasets, which no overlap on the device hides).
static bool slab_contiguous(int32_t count, gprb_dataset* const* ds, const double* const* X, int64_t ldx) {
  if (count < 1 || !ds[0]->slab || ds[0]->slab->count != count || ldx != ds[0]->d) return false;
  for (int i = 0; i < count; ++i) {
    if (ds[i]->slab != ds[0]->slab || ds[i]->slab_index != i) return false;
    if (X[i] != X[0] + (int64_t)i * ds[0]->n * ldx) return false;
  }
  return true;
}

static int slab_upload(gprb_ctx* ctx, int32_t count, gprb_dataset* const* ds, const double* X0) {
  gprb_slab* sl = ds[0]->slab;
  const int64_t n = ds[0]->n, npad = ds[0]->npad;
  const int d = ds[0]->d;
  for (int i = 0; i < count; ++i) ds[i]->version++;
  GPRB_CUDA(cudaMemcpyAsync(sl->X, X0, sizeof(double) * (size_t)count * n * d, cudaMemcpyHostToDevice, ctx->upload));
  int rc = launch_transpose_inputs_batched(sl->X, sl->Xt, (int)n, (int)npad, d, count, ctx->upload);
  if (rc) return rc;
  ctx->launches++;
  GPRB_CUDA(cudaStreamSynchronize(ctx->upload));
  return 0;
}

int gprb_datasets_create(gprb_ctx* ctx, int32_t count, int64_t n, int32_t d, const double* const* X, int64_t ldx,
                         gprb_dataset** out) {
  GPRB_REQUIRE(ctx && X && out && count >= 1, "gprb_datasets_create: bad argument");
  GPRB_REQUIRE(n >= 1 && n <= (1 << 20), "gprb_datasets_create: n out of range");
  GPRB_REQUIRE(d >= 1 && d <= MAX_D, "gprb_datasets_create: d must be in 1..62");
  GPRB_REQUIRE(ldx >= d, "gprb_datasets_create: ldx < d");
  for (int i = 0; i < count; ++i) { GPRB_REQUIRE(X[i] != nullptr, "gprb_datasets_create: NULL matrix"); out[i] = nullptr; }
  GPRB_CUDA(cudaSetDevice(ctx->device));
  const int64_t npad = (n + NB - 1) / NB * NB;
  gprb_slab* sl = new (std::nothrow) gprb_slab();
  GPRB_REQUIRE(sl != nullptr, "gprb_datasets_create: out of host memory");
  int rc;
  if ((rc = dev_alloc(&sl->X, (size_t)count * n * d)) || (rc = dev_alloc(&sl->Xt, (size_t)count * npad * d))) {
    cudaFree(sl->X); cudaFree(sl->Xt); delete sl;
    return rc;
  }
  sl->count = count; sl->refs = count;
  for (int i = 0; i < count; ++i) {
    gprb_dataset* ds = new (std::nothrow) gprb_dataset();
    if (!ds) {  // unwind
      for (int k = 0; k < i; ++k) { delete out[k]; out[k] = nullptr; }
      cudaFree(sl->X); cudaFree(sl->Xt); delete sl;
      set_error("gprb_datasets_create: out of host memory");
      return GPRB_ERR_ARG;
    }
    ds->ctx = ctx; ds->n = n; ds->d = d; ds->npad = npad;
    ds->X = sl->X + (size_t)i * n * d;
    ds->Xt = sl->Xt + (size_t)i * npad * d;
    ds->slab = sl; ds->slab_index = i;
    out[i] = ds;
  }
  rc = gprb_datasets_update(ctx, count, out, X, ldx);
  if (rc) {
    for (int i = 0; i < count; ++i) { delete out[i]; out[i] = nullptr; }
    cudaFree(sl->X); cudaFree(sl->Xt); delete sl;
  }
  return rc;
}

int gprb_datasets_update(gprb_ctx* ctx, int32_t count, gprb_dataset* const* ds, const double* const* X, int64_t ldx) {
  GPRB_REQUIRE(ctx && ds && X && count >= 0, "gprb_datasets_update: bad argument");
  for (int i = 0; i < count; ++i) {
    GPRB_REQUIRE(ds[i] && X[i], "gprb_datasets_update: NULL dataset or matrix");
    GPRB_REQUIRE(ds[i]->ctx == ctx, "gprb_datasets_update: dataset belongs to another context");
    GPRB_REQUIRE(ldx >= ds[i]->d, "gprb_datasets_update: ldx < d");
  }
  GPRB_CUDA(cudaSetDevice(ctx->device));
  if (slab_contiguous(count, ds, X, ldx)) return slab_upload(ctx, count, ds, X[0]);
  // The copies are queued back to back on the upload stream (truly asynchronous when the host matrices are page-locked);
  // the transposes run on a second stream, a quarter of the datasets at a time, behind an event - a transpose between
  // two copies on one stream would stall the copy engine for a kernel launch each time (2.6 -> 1.4 ms per 100 datasets).
  // One synchronisation at the end keeps the "synchronous on return" contract.
  const int chunk = std::max(1, (count + 3) / 4);
  for (int i0 = 0; i0 < count; i0 += chunk) {
    const int i1 = std::min(count, i0 + chunk);
    for (int i = i0; i < i1; ++i) {
      int rc = dataset_copy_async(ds[i], X[i], ldx, ctx->upload);
      if (rc) return rc;
    }
    GPRB_CUDA(cudaEventRecord(ctx->upload_ev, ctx->upload));
    GPRB_CUDA(cudaStreamWaitEvent(ctx->upload2, ctx->upload_ev, 0));
    for (int i = i0; i < i1; ++i) {
      int rc = launch_transpose_inputs(ds[i]->X, ds[i]->Xt, (int)ds[i]->n, (int)ds[i]->npad, ds[i]->d, ctx->upload2);
      if (rc) return rc;
      ctx->launches++;
    }
  }
  GPRB_CUDA(cudaStreamSynchronize(ctx->upload));
  GPRB_CUDA(cudaStreamSynchronize(ctx->upload2));
  return GPRB_OK;
}

int gprb_dataset_destroy(gprb_dataset* ds) {
  if (!ds) return GPRB_OK;
  if (ds->slab) {
    if (--ds->slab->refs == 0) {
      cudaSetDevice(ds->ctx->device);
      cudaFree(ds->slab->X); cudaFree(ds->slab->Xt);
      delete ds->slab;
    }
  } else {
    cudaFree(ds->X); cudaFree(ds->Xt);
  }
  delete ds;
  return GPRB_OK;
}

// ------------------------------------------------------------------------------------------------
static int upload_targets(gprb_batch* b, const double* ymm) {
  GPRB_CUDA(cudaMemcpy2DAsync(b->ymm, sizeof(double) * b->npad, ymm, sizeof(double) * b->n, sizeof(double) * b->n, b->B,
                              cudaMemcpyHostToDevice, b->stream[0]));
  GPRB_CUDA(cudaStreamSynchronize(b->stream[0]));
  b->state_ok.assign(b->B, 0);
  b->inv_ok.assign(b->B, 0);
  b->v_ok.assign(b->B, 0);
  return 0;
}

int gprb_batch_create(gprb_ctx* ctx, int32_t B, gprb_dataset* const* ds, const double* ymm, int32_t kernel_kind,
                      gprb_batch** out) {
  GPRB_REQUIRE(ctx && ds && ymm && out, "gprb_batch_create: NULL argument");
  *out = nullptr;
  GPRB_REQUIRE(B >= 1 && B <= 65535, "gprb_batch_create: B must be in 1..65535");
  GPRB_REQUIRE(kernel_kind >= 0 && kernel_kind <= 3, "gprb_batch_create: unknown kernel_kind");
  for (int i = 0; i < B; ++i) {
    GPRB_REQUIRE(ds[i] != nullptr, "gprb_batch_create: NULL dataset");
    GPRB_REQUIRE(ds[i]->ctx == ctx, "gprb_batch_create: dataset belongs to another context");
    GPRB_REQUIRE(ds[i]->n == ds[0]->n && ds[i]->d == ds[0]->d, "gprb_batch_create: datasets differ in n or d");
  }
  GPRB_CUDA(cudaSetDevice(ctx->device));
  gprb_batch* b = new (std::nothrow) gprb_batch();
  GPRB_REQUIRE(b != nullptr, "gprb_batch_create: out of host memory");
  b->ctx = ctx; b->B = B; b->n = ds[0]->n; b->d = ds[0]->d; b->P = b->d + 2; b->kind = kernel_kind;
  b->npad = ds[0]->npad; b->J = (int)(b->npad / NB);
  b->ds.assign(ds, ds + B);
  for (gprb_dataset* u : distinct_datasets(b)) u->users++;
  const size_t mat = (size_t)b->npad * b->npad, dinv = (size_t)b->J * NB * NB;
  const size_t ntiles = (size_t)b->J * (b->J + 1) / 2;
  int rc = 0;
  do {
    if ((rc = dev_alloc(&b->Xptr, B)) || (rc = dev_alloc(&b->Xtptr, B)) || (rc = dev_alloc(&b->ymm, (size_t)B * b->npad)) ||
        (rc = dev_alloc(&b->theta, (size_t)B * b->P)) || (rc = dev_alloc(&b->A, mat * B)) || (rc = dev_alloc(&b->Lm, mat * B)) ||
        (rc = dev_alloc(&b->Dinv, dinv * B)) || (rc = dev_alloc(&b->DinvT, dinv * B)) || (rc = dev_alloc(&b->KinvD, dinv * B)) ||
        (rc = dev_alloc(&b->alpha, (size_t)B * b->npad)) || (rc = dev_alloc(&b->zbuf, (size_t)B * b->npad)) ||
        (rc = dev_alloc(&b->jitter, B)) || (rc = dev_alloc(&b->diag_off, B)) || (rc = dev_alloc(&b->logdet_part, (size_t)B * b->J)) ||
        (rc = dev_alloc(&b->fail, B)) || (rc = dev_alloc(&b->mll, B)) || (rc = dev_alloc(&b->grad, (size_t)B * b->P)) ||
        (rc = dev_alloc(&b->grad_part, (size_t)B * ntiles * GRAD_PARTS_PER_TILE * b->P)) || (rc = dev_alloc(&b->list, 2 * (size_t)B)))
      break;
    b->stage_doubles = (int64_t)B * (b->P + 2);
    cudaError_t e;
    if ((e = cudaMallocHost((void**)&b->list_host, sizeof(int32_t) * 2 * B)) != cudaSuccess ||
        (e = cudaMallocHost((void**)&b->fail_host, sizeof(int32_t) * B)) != cudaSuccess ||
        (e = cudaMallocHost((void**)&b->stage_host, sizeof(double) * b->stage_doubles)) != cudaSuccess) {
      rc = cuda_fail(e, "cudaMallocHost", __FILE__, __LINE__);
      break;
    }
    if ((rc = set_batch_gemm(b))) break;
    b->nstreams = 4;
    b->rl_max = 24;
    if (const char* ev = getenv("GPRB200_RL_MAX")) b->rl_max = atoi(ev);
    // launches of the substitution with at most a quarter of the SM count in GPs (<= 37 on a B200: the reference's per-GP
    // call pattern, straggler rounds of the optimiser, the stream groups of the 8-GPU strong split) run one thread-block
    // cluster per GP; above that the one-CTA-per-GP kernel already streams at the HBM roof and clusters only add barriers
    // (measured: 100-GP groups, 122.0 -> 129.2 ms per 400-GP step with clusters)
    b->solve_cluster_below = ctx->sm_count / 4 + 1;
    b->group_skew = 0.0;
    if (const char* ev = getenv("GPRB200_GROUP_SKEW")) b->group_skew = std::max(0.0, std::min(0.9, atof(ev)));
    if (const char* ev = getenv("GPRB200_SOLVE_CLUSTER_BELOW")) b->solve_cluster_below = atoi(ev);
    if (const char* ev = getenv("GPRB200_STREAMS")) b->nstreams = std::max(1, std::min(MAX_STREAMS, atoi(ev)));
    for (int s = 0; s < MAX_STREAMS && !rc; ++s) {
      if ((e = cudaStreamCreateWithFlags(&b->stream[s], cudaStreamNonBlocking)) != cudaSuccess ||
          (e = cudaEventCreateWithFlags(&b->join[s], cudaEventDisableTiming)) != cudaSuccess)
        rc = cuda_fail(e, "stream/event create", __FILE__, __LINE__);
    }
    for (int s = 0; s < 8 && !rc; ++s)
      if ((e = cudaEventCreate(&b->ev[s])) != cudaSuccess) rc = cuda_fail(e, "cudaEventCreate", __FILE__, __LINE__);
    if (rc) break;
    std::vector<const double*> xp(B), xtp(B);
    for (int i = 0; i < B; ++i) { xp[i] = ds[i]->X; xtp[i] = ds[i]->Xt; }
    if ((e = cudaMemcpy(b->Xptr, xp.data(), sizeof(double*) * B, cudaMemcpyHostToDevice)) != cudaSuccess ||
        (e = cudaMemcpy(b->Xtptr, xtp.data(), sizeof(double*) * B, cudaMemcpyHostToDevice)) != cudaSuccess ||
        (e = cudaMemset(b->theta, 0, sizeof(double) * B * b->P)) != cudaSuccess ||
        (e = cudaMemset(b->jitter, 0, sizeof(double) * B)) != cudaSuccess ||
        (e = cudaMemset(b->diag_off, 0, sizeof(double) * B)) != cudaSuccess ||
        (e = cudaMemset(b->ymm, 0, sizeof(double) * b->npad * B)) != cudaSuccess ||  // zero padding, written once
        (e = cudaMemset(b->fail, 0, sizeof(int32_t) * B)) != cudaSuccess ||
        // k_diag_factor only writes the triangular halves of the inverted diagonal blocks: the zero halves are set here
        (e = cudaMemset(b->Dinv, 0, sizeof(double) * dinv * B)) != cudaSuccess ||
        (e = cudaMemset(b->DinvT, 0, sizeof(double) * dinv * B)) != cudaSuccess) {
      rc = cuda_fail(e, "batch init copies", __FILE__, __LINE__);
      break;
    }
    rc = upload_targets(b, ymm);
  } while (0);
  if (rc) {
    for (gprb_dataset* u : distinct_datasets(b)) u->users--;
    free_batch(b);
    return rc;
  }
  *out = b;
  return GPRB_OK;
}

int gprb_batch_set_targets(gprb_batch* b, const double* ymm) {
  GPRB_REQUIRE(b && ymm, "gprb_batch_set_targets: NULL argument");
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  return upload_targets(b, ymm);
}

int gprb_batch_set_diag_offset(gprb_batch* b, const double* offset) {
  GPRB_REQUIRE(b, "gprb_batch_set_diag_offset: NULL batch");
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  if (offset) {
    for (int i = 0; i < b->B; ++i) GPRB_REQUIRE(isfinite(offset[i]), "gprb_batch_set_diag_offset: non-finite offset");
    GPRB_CUDA(cudaMemcpy(b->diag_off, offset, sizeof(double) * b->B, cudaMemcpyHostToDevice));
  } else {
    GPRB_CUDA(cudaMemset(b->diag_off, 0, sizeof(double) * b->B));
  }
  // a different matrix is factorised from now on: nothing resident may be reused
  b->state_ok.assign(b->B, 0); b->inv_ok.assign(b->B, 0); b->v_ok.assign(b->B, 0);
  std::fill(b->theta_valid.begin(), b->theta_valid.end(), (uint8_t)0);
  return GPRB_OK;
}

int gprb_batch_destroy(gprb_batch* b) {
  if (b) {
    cudaSetDevice(b->ctx->device);
    cudaDeviceSynchronize();
    for (gprb_dataset* u : distinct_datasets(b)) u->users--;
  }
  free_batch(b);
  return GPRB_OK;
}

int gprb_set_profiling(gprb_batch* b, int32_t on) {
  GPRB_REQUIRE(b, "gprb_set_profiling: NULL batch");
  b->profiling = on != 0;
  return GPRB_OK;
}

int gprb_last_gemm_launch_ms(gprb_batch* b, double* out, int32_t cap) {
  GPRB_REQUIRE(b && (out || cap == 0), "gprb_last_gemm_launch_ms: NULL argument");
  const int n = (int)b->gemm_ms.size();
  for (int i = 0; i < n && i < cap; ++i) out[i] = b->gemm_ms[i];
  return n;
}

int gprb_last_stage_ms(gprb_batch* b, double out[8]) {
  GPRB_REQUIRE(b && out, "gprb_last_stage_ms: NULL argument");
  for (int i = 0; i < 8; ++i) out[i] = b->stage_ms[i];
  return GPRB_OK;
}

// ------------------------------------------------------------------------------------------------
int gprb_eval_mixed(gprb_batch* b, const double* theta, const uint8_t* mode, double* mll, double* grad, int32_t* info) {
  GPRB_REQUIRE(b && theta && mode && mll && info, "gprb_eval_mixed: NULL argument");
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  bool any_grad = false;
  std::vector<int32_t> act;
  for (int i = 0; i < b->B; ++i) {
    GPRB_REQUIRE(mode[i] <= 2, "gprb_eval_mixed: mode must be 0 (skip), 1 (value) or 2 (value+gradient)");
    if (mode[i]) act.push_back(i);
    any_grad = any_grad || mode[i] == 2;
  }
  GPRB_REQUIRE(!any_grad || grad, "gprb_eval_mixed: a GP asks for its gradient but grad is NULL");
  int rc = upload_theta_rows(b, theta, act);
  if (rc) return rc;
  std::vector<int32_t> inf;
  if ((rc = evaluate_modes(b, theta, mode, inf))) return rc;
  return download_results(b, mode, inf, nullptr, mll, grad, info);
}

int gprb_eval(gprb_batch* b, const double* theta, const uint8_t* active, double* mll, double* grad, int32_t* info) {
  GPRB_REQUIRE(b && theta && mll && info, "gprb_eval: NULL argument");
  std::vector<uint8_t> mode(b->B);
  for (int i = 0; i < b->B; ++i) mode[i] = (!active || active[i]) ? (grad ? 2 : 1) : 0;
  return gprb_eval_mixed(b, theta, mode.data(), mll, grad, info);
}

int gprb_eval_device(gprb_batch* b, const double* theta_dev, double* mll_dev, double* grad_dev, int32_t* info_dev,
                     void* stream) {
  GPRB_REQUIRE(b && theta_dev && mll_dev, "gprb_eval_device: NULL argument");
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  cudaStream_t user = (cudaStream_t)stream;
  const int B = b->B, P = b->P;
  // order after the caller's stream, run on the batch streams, hand results back on the caller's stream
  GPRB_CUDA(cudaEventRecord(b->join[0], user));
  GPRB_CUDA(cudaStreamWaitEvent(b->stream[0], b->join[0], 0));
  GPRB_CUDA(cudaMemcpyAsync(b->theta, theta_dev, sizeof(double) * B * P, cudaMemcpyDeviceToDevice, b->stream[0]));
  std::vector<uint8_t> mode(B, grad_dev ? 2 : 1);
  std::vector<int32_t> inf;
  int rc = evaluate_modes(b, nullptr, mode.data(), inf);  // theta lives on the device: nothing to compare, nothing remembered
  if (rc) return rc;
  GPRB_CUDA(cudaMemcpyAsync(mll_dev, b->mll, sizeof(double) * B, cudaMemcpyDeviceToDevice, b->stream[0]));
  if (grad_dev) GPRB_CUDA(cudaMemcpyAsync(grad_dev, b->grad, sizeof(double) * B * P, cudaMemcpyDeviceToDevice, b->stream[0]));
  if (info_dev) {
    memcpy(b->fail_host, inf.data(), sizeof(int32_t) * B);
    GPRB_CUDA(cudaMemcpyAsync(info_dev, b->fail_host, sizeof(int32_t) * B, cudaMemcpyHostToDevice, b->stream[0]));
  }
  GPRB_CUDA(cudaEventRecord(b->join[0], b->stream[0]));
  GPRB_CUDA(cudaStreamWaitEvent(user, b->join[0], 0));
  GPRB_CUDA(cudaStreamSynchronize(b->stream[0]));
  return GPRB_OK;
}

// ------------------------------------------------------------------------------------------------
}  // extern "C"

template <typename T>
static int ensure_dev(T** p, size_t* cap, size_t need, bool zero = false) {
  if (*p && *cap >= need) return 0;
  cudaFree(*p);
  *p = nullptr; *cap = 0;
  int rc = dev_alloc(p, need);
  if (rc) return rc;
  if (zero) GPRB_CUDA(cudaMemset(*p, 0, sizeof(T) * need));
  *cap = need;
  return 0;
}

static int ensure_pinned(double** p, size_t* cap, size_t need) {
  if (*p && *cap >= need) return 0;
  if (*p) cudaFreeHost(*p);
  *p = nullptr; *cap = 0;
  cudaError_t e = cudaMallocHost((void**)p, sizeof(double) * std::max<size_t>(need, 1));
  if (e != cudaSuccess) return cuda_fail(e, "cudaMallocHost(predict staging)", __FILE__, __LINE__);
  *cap = need;
  return 0;
}

// Stage a prediction of the GPs gp0 .. gp1-1 (one Xstar block per gpb consecutive GPs) on pipeline `slot`: the slot's
// events and mask on first use, grow-only scratch (h_out: h_out_doubles), the per-GP mask, the inputs through the pinned
// staging; then t0 and the uploads on the slot's first stream.
static int predict_stage(gprb_batch* b, int slot, int gp0, int gp1, int gpb, int64_t m, const double* Xstar,
                         int64_t xstar_stride, const double* mstar, size_t h_out_doubles) {
  gprb_predict_slot& sl = b->ps[slot];
  const int B = b->B, count = gp1 - gp0;
  cudaStream_t st = b->stream[4 * slot];
  const int nblocks = (count + gpb - 1) / gpb;  // Xstar blocks: one per gpb consecutive GPs (the outputs of a trial)
  const size_t nx = (size_t)(xstar_stride ? xstar_stride * (nblocks - 1) + m * b->d : m * b->d);
  const size_t nout = (size_t)count * m;
  int rc;
  if (!sl.t0) {
    GPRB_CUDA(cudaEventCreate(&sl.t0));
    GPRB_CUDA(cudaEventCreate(&sl.t1));
    GPRB_CUDA(cudaMallocHost((void**)&sl.h_mask, sizeof(int32_t) * B));
    if ((rc = dev_alloc(&sl.mask, (size_t)B))) return rc;
  }
  if ((rc = ensure_dev(&sl.pX, &sl.pX_cap, nx)) || (rc = ensure_dev(&sl.pmu, &sl.pmu_cap, nout)) ||
      (rc = ensure_pinned(&sl.h_in, &sl.h_in_cap, nx + (mstar ? nout : 0))) ||
      (rc = ensure_pinned(&sl.h_out, &sl.h_out_cap, h_out_doubles)))
    return rc;
  if (mstar && (rc = ensure_dev(&sl.pms, &sl.pms_cap, nout))) return rc;
  // per-GP mask: a GP without an evaluated state gets NaN rows and blocks nobody (examples/parallel/core.jl:41-46)
  for (int i = 0; i < B; ++i) sl.h_mask[i] = b->state_ok[i] ? 0 : 1;
  memcpy(sl.h_in, Xstar, sizeof(double) * nx);
  if (mstar) memcpy(sl.h_in + nx, mstar, sizeof(double) * nout);
  GPRB_CUDA(cudaEventRecord(sl.t0, st));
  GPRB_CUDA(cudaMemcpyAsync(sl.mask, sl.h_mask, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
  GPRB_CUDA(cudaMemcpyAsync(sl.pX, sl.h_in, sizeof(double) * nx, cudaMemcpyHostToDevice, st));
  if (mstar) GPRB_CUDA(cudaMemcpyAsync(sl.pms, sl.h_in + nx, sizeof(double) * nout, cudaMemcpyHostToDevice, st));
  return 0;
}

// The slot's right-hand-side block pT [count][npad][PT] and its tensor map (row r = k, box = 68 columns x KT rows),
// re-encoded whenever pT is (re)allocated.
static int slot_rhs(gprb_batch* b, gprb_predict_slot& sl, int count) {
  int rc;
  if ((rc = ensure_dev(&sl.pT, &sl.pT_cap, (size_t)count * b->npad * PT))) return rc;
  if (sl.tm_T_cap != sl.pT_cap) {
    if ((rc = make_tensor_map(&sl.tm_T68, sl.pT, PT, (uint64_t)b->npad, sl.pT_cap / ((size_t)b->npad * PT), PT, (uint64_t)b->npad * PT,
                              NB / 2 + 4, KT)))
      return rc;
    sl.tm_T_cap = sl.pT_cap;
  }
  return 0;
}

// One dependent chain of J tile-GEMM launches, one per block row: GEMM_FWD_ROW top-down, GEMM_BWD_ROW bottom-up.
static int row_chain(gprb_batch* b, GemmArgs& ga, int mode, int ntl, int count, cudaStream_t st) {
  ga.mode = mode;
  for (int k = 0; k < ga.J; ++k) {
    ga.step = mode == GEMM_BWD_ROW ? ga.J - 1 - k : k;
    if (int rc = launch_tile_gemm(ga, ntl, count, st)) return rc;
    b->ctx->launches++;
  }
  return 0;
}

// The tiled path of a prediction staged on `slot` (predict_stage), one chunk of PT test columns at a time:
// k_predict_cross on the slot's first stream; the GPs dealt over stream groups (the slot's streams and join events),
// each of which runs the FWD_ROW chain T = L^-1 K* when T != nullptr and then hook(ta, ga, ntl, g0, g1, stream) on its
// stream; with `finish`, k_predict_finish of the whole range on the slot's first stream.  T is [count][npad][PT] behind
// tm_T, or with keep_T one such block per chunk (chunk c of local GP g is block c * count + g).  hook = nullptr: no
// per-group work besides the chain.
template <typename Hook>
static int predict_tiles(gprb_batch* b, int slot, int gp0, int gp1, int gpb, int64_t m, int64_t xstar_stride, bool mstar,
                         double* var, double* T, const CUtensorMap& tm_T, bool keep_T, bool finish, Hook&& hook) {
  constexpr bool has_hook = !std::is_same<Hook, std::nullptr_t>::value;
  static const char* zmax = getenv("GPRB200_PC_ZMAX");
  gprb_predict_slot& sl = b->ps[slot];
  const int J = b->J, count = gp1 - gp0;
  const int64_t npad = b->npad;
  cudaStream_t* str = b->stream + 4 * slot;
  cudaEvent_t* join = b->join + 4 * slot;
  int rc;
  if ((rc = ensure_dev(&sl.pmupart, &sl.pmupart_cap, (size_t)count * J * PT))) return rc;
  // L^-1 K*: one launch per block row, `count` tiles of 128 x 128 each (PDMats whiten! as a blocked substitution)
  GemmArgs ga = b->gemm;
  ga.Cin = nullptr;
  ga.Tm = T; ga.t_stride = npad * PT; ga.ldt = PT;
  ga.tm_T68 = tm_T;
  ga.fail = sl.mask;  // tiles of a GP without state exit at once
  // the GPs are dealt over the stream groups: the dependent chain of J launches of one group fills the wave
  // tails of the others (`count` tiles per launch are not a multiple of the SM count); with no work per group (a
  // mean-only gprb_predict) there is one group and no event
  const int ns = std::min(4, b->nstreams);
  const int S = (T || has_hook) && count >= 8 * ns ? ns : 1;
  for (int c = 0; (int64_t)c * PT < m; ++c) {
    const int64_t s0 = (int64_t)c * PT;
    const int tblk = keep_T ? c * count : 0;  // T block of the chunk's first GP
    PredictTileArgs ta{b->Xtptr, b->theta, b->alpha, sl.pX, mstar ? sl.pms : nullptr, T ? T + (size_t)tblk * npad * PT : nullptr,
                       sl.pmupart, sl.pmu, var, xstar_stride, (int)b->n, (int)npad, b->d, J, (int)m, b->kind, (int)s0,
                       (int)std::min<int64_t>(PT, m - s0)};
    ta.gp_off = gp0;
    ta.mask = sl.mask;
    ta.gpb = gpb;
    if (zmax) ta.zmax = atof(zmax);
    if ((rc = launch_predict_cross(ta, count, str[0]))) return rc;
    b->ctx->launches++;
    ga.t_gp_off = gp0 - tblk;
    ga.ncols = ta.mc;
    // right-hand-side tiles are 64 test columns wide (two CTAs per SM); few GPs (large n, or the reference's single-GP
    // call pattern): 32-column tiles, so that a launch still puts a CTA on every SM
    ga.colw = (int64_t)count * ((ta.mc + 63) / 64) >= b->ctx->sm_count ? 64 : 32;
    const int ntl = (ta.mc + ga.colw - 1) / ga.colw;
    if (S > 1) GPRB_CUDA(cudaEventRecord(join[0], str[0]));
    for (int s = 0; s < S; ++s) {
      const int g0 = (int)((int64_t)count * s / S), g1 = (int)((int64_t)count * (s + 1) / S);
      if (s > 0) GPRB_CUDA(cudaStreamWaitEvent(str[s], join[0], 0));
      ga.gp_off = gp0 + g0;
      if (T && (rc = row_chain(b, ga, GEMM_FWD_ROW, ntl, g1 - g0, str[s]))) return rc;
      if constexpr (has_hook)
        if ((rc = hook(ta, ga, ntl, g0, g1, str[s]))) return rc;
      if (s > 0) {
        GPRB_CUDA(cudaEventRecord(join[s], str[s]));
        GPRB_CUDA(cudaStreamWaitEvent(str[0], join[s], 0));
      }
    }
    if (finish) {
      if ((rc = launch_predict_finish(ta, count, str[0]))) return rc;
      b->ctx->launches++;
    }
  }
  return 0;
}

// Wait for the slot's t1 and keep the device time t0 .. t1 of its last call (gprb_last_predict_ms).
static int slot_wait(gprb_predict_slot& sl) {
  GPRB_CUDA(cudaEventSynchronize(sl.t1));
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, sl.t0, sl.t1) == cudaSuccess) sl.last_ms = ms;
  return 0;
}

// Enqueue the prediction of the GPs gp0 .. gp1-1 on pipeline `slot` (streams 4 slot .. 4 slot + 3): inputs are copied to
// the slot's pinned staging, everything else is asynchronous; predict_collect waits and hands the results out.
static int predict_enqueue(gprb_batch* b, int slot, int gp0, int gp1, int64_t m, const double* Xstar, int64_t xstar_stride,
                           const double* mstar, bool want_var, int gpb = 1) {
  gprb_predict_slot& sl = b->ps[slot];
  const int J = b->J, count = gp1 - gp0;
  cudaStream_t st = b->stream[4 * slot];
  const size_t nout = (size_t)count * m;
  int rc;
  if ((rc = predict_stage(b, slot, gp0, gp1, gpb, m, Xstar, xstar_stride, mstar, 2 * nout))) return rc;
  if (want_var && (rc = ensure_dev(&sl.pvar, &sl.pvar_cap, nout))) return rc;
  bool all_v = true, any_ok = false;
  for (int i = gp0; i < gp1; ++i)
    if (b->state_ok[i]) { any_ok = true; all_v = all_v && b->v_ok[i]; }

  // GEMV-like path: few test columns and the triangular inverse already resident (the last evaluation had a gradient)
  const int ps = m <= 1 ? 1 : m <= 2 ? 2 : m <= 4 ? 4 : 8;
  const size_t small_smem = ((size_t)ps * b->npad + ps * MAX_D + MAX_D + 8) * sizeof(double);
  if (want_var && m <= 8 && all_v && any_ok && small_smem <= 227 * 1024) {
    const int ncc = (int)((m + ps - 1) / ps);
    // CTAs sharing the row chunks of one (GP, column chunk): enough to put ~2 CTAs on every SM, a power of two <= 16
    int rs = 1;
    while (rs < PRED_CHUNKS && (int64_t)count * ncc * rs < 2 * (int64_t)b->ctx->sm_count) rs *= 2;
    if ((rc = ensure_dev(&sl.pq, &sl.pq_cap, (size_t)count * ncc * PRED_CHUNKS * 16)) ||
        (rc = ensure_dev(&sl.pcount, &sl.pcount_cap, (size_t)count * ncc, true)))
      return rc;
    PredictArgs pa{b->Xptr, b->theta, b->alpha, b->Lm, b->DinvT, sl.pX, mstar ? sl.pms : nullptr, sl.pmu, sl.pvar,
                   sl.pq, sl.pcount, sl.mask, xstar_stride, b->npad * b->npad, (int64_t)J * NB * NB,
                   (int)b->n, (int)b->npad, b->d, (int)m, b->kind, gp0, rs, gpb};
    if ((rc = launch_predict(pa, count, st))) return rc;
    b->ctx->launches++;
  } else {
    if (want_var && (rc = slot_rhs(b, sl, count))) return rc;
    if ((rc = predict_tiles(b, slot, gp0, gp1, gpb, m, xstar_stride, mstar != nullptr, want_var ? sl.pvar : nullptr,
                            want_var ? sl.pT : nullptr, sl.tm_T68, false, true, nullptr)))
      return rc;
  }
  GPRB_CUDA(cudaMemcpyAsync(sl.h_out, sl.pmu, sizeof(double) * nout, cudaMemcpyDeviceToHost, st));
  if (want_var) GPRB_CUDA(cudaMemcpyAsync(sl.h_out + nout, sl.pvar, sizeof(double) * nout, cudaMemcpyDeviceToHost, st));
  GPRB_CUDA(cudaEventRecord(sl.t1, st));
  sl.pending = true; sl.gp0 = gp0; sl.gp1 = gp1; sl.m = m; sl.want_var = want_var;
  return 0;
}

static int predict_collect(gprb_batch* b, int slot, double* mu, double* var) {
  gprb_predict_slot& sl = b->ps[slot];
  int rc = slot_wait(sl);
  if (rc) return rc;
  sl.pending = false;
  const size_t nout = (size_t)(sl.gp1 - sl.gp0) * sl.m;
  memcpy(mu, sl.h_out, sizeof(double) * nout);
  if (var && sl.want_var) memcpy(var, sl.h_out + nout, sizeof(double) * nout);
  return 0;
}

static int predict_check(gprb_batch* b, int slot, int gp0, int gp1, int64_t m, const double* Xstar, int64_t xstar_stride) {
  GPRB_REQUIRE(b && Xstar, "gprb_predict: NULL argument");
  GPRB_REQUIRE(slot == 0 || slot == 1, "gprb_predict: slot must be 0 or 1");
  GPRB_REQUIRE(gp0 >= 0 && gp0 < gp1 && gp1 <= b->B, "gprb_predict: bad GP range");
  GPRB_REQUIRE(m >= 1 && m <= (1 << 24), "gprb_predict: m out of range");
  GPRB_REQUIRE(xstar_stride == 0 || xstar_stride >= m * b->d, "gprb_predict: xstar_stride must be 0 or >= d*m");
  GPRB_REQUIRE(!b->ps[slot].pending, "gprb_predict: the slot has a prediction in flight - call gprb_predict_wait first");
  return 0;
}

extern "C" {

int gprb_predict(gprb_batch* b, int64_t m, const double* Xstar, int64_t xstar_stride, const double* mstar, double* mu,
                 double* var) {
  GPRB_REQUIRE(b && mu, "gprb_predict: NULL argument");
  int rc = predict_check(b, 0, 0, b->B, m, Xstar, xstar_stride);
  if (rc) return rc;
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  if ((rc = predict_enqueue(b, 0, 0, b->B, m, Xstar, xstar_stride, mstar, var != nullptr))) return rc;
  return predict_collect(b, 0, mu, var);
}

int gprb_predict_async(gprb_batch* b, int32_t slot, int32_t gp0, int32_t gp1, int64_t m, const double* Xstar,
                       int64_t xstar_stride, int32_t gps_per_block, const double* mstar, int32_t want_var) {
  int rc = predict_check(b, slot, gp0, gp1, m, Xstar, xstar_stride);
  if (rc) return rc;
  GPRB_REQUIRE(gps_per_block >= 1, "gprb_predict_async: gps_per_block must be >= 1");
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  return predict_enqueue(b, slot, gp0, gp1, m, Xstar, xstar_stride, mstar, want_var != 0, gps_per_block);
}

int gprb_predict_wait(gprb_batch* b, int32_t slot, double* mu, double* var) {
  GPRB_REQUIRE(b && mu && (slot == 0 || slot == 1), "gprb_predict_wait: bad argument");
  GPRB_REQUIRE(b->ps[slot].pending, "gprb_predict_wait: no prediction in flight on this slot");
  GPRB_REQUIRE(!var || b->ps[slot].want_var, "gprb_predict_wait: var requested but the prediction was enqueued with want_var = 0");
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  return predict_collect(b, slot, mu, var);
}

int gprb_last_predict_ms(gprb_batch* b, int32_t slot, double* ms) {
  GPRB_REQUIRE(b && ms && (slot == 0 || slot == 1), "gprb_last_predict_ms: bad argument");
  *ms = b->ps[slot].last_ms;
  return GPRB_OK;
}

// ------------------------------------------------------------------------------------------------
static int fetch_matrix(gprb_batch* b, const double* dev, std::vector<double>& host) {
  host.resize((size_t)b->npad * b->npad);
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  GPRB_CUDA(cudaStreamSynchronize(b->stream[0]));
  GPRB_CUDA(cudaMemcpy(host.data(), dev, sizeof(double) * host.size(), cudaMemcpyDeviceToHost));
  return 0;
}

int gprb_get_K(gprb_batch* b, int32_t gp, double* out) {
  GPRB_REQUIRE(b && out && gp >= 0 && gp < b->B, "gprb_get_K: bad argument");
  GPRB_REQUIRE(b->state_ok[gp], "gprb_get_K: no evaluated state");
  // K (noise and make_posdef! jitter included) stays resident in the lower tiles of A through every stage
  std::vector<double> h;
  int rc = fetch_matrix(b, b->A + (size_t)gp * b->npad * b->npad, h);
  if (rc) return rc;
  const int64_t n = b->n, np = b->npad;
  for (int64_t c = 0; c < n; ++c)
    for (int64_t r = c; r < n; ++r) out[r + c * n] = out[c + r * n] = h[r + c * np];
  return GPRB_OK;
}

int gprb_get_chol(gprb_batch* b, int32_t gp, double* out) {
  GPRB_REQUIRE(b && out && gp >= 0 && gp < b->B, "gprb_get_chol: bad argument");
  GPRB_REQUIRE(b->state_ok[gp], "gprb_get_chol: no evaluated state");
  std::vector<double> h;
  int rc = fetch_matrix(b, b->Lm + (size_t)gp * b->npad * b->npad, h);
  if (rc) return rc;
  const int64_t n = b->n, np = b->npad;
  for (int64_t c = 0; c < n; ++c)
    for (int64_t r = 0; r < n; ++r) out[r + c * n] = (r <= c) ? h[c + r * np] : 0.0;  // U(r,c) = L(c,r)
  return GPRB_OK;
}

int gprb_get_alpha(gprb_batch* b, int32_t gp, double* out) {
  GPRB_REQUIRE(b && out && gp >= 0 && gp < b->B, "gprb_get_alpha: bad argument");
  GPRB_REQUIRE(b->state_ok[gp], "gprb_get_alpha: no evaluated state");
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  GPRB_CUDA(cudaStreamSynchronize(b->stream[0]));
  GPRB_CUDA(cudaMemcpy(out, b->alpha + (size_t)gp * b->npad, sizeof(double) * b->n, cudaMemcpyDeviceToHost));
  return GPRB_OK;
}

int gprb_get_Kinv(gprb_batch* b, int32_t gp, double* out) {
  GPRB_REQUIRE(b && out && gp >= 0 && gp < b->B, "gprb_get_Kinv: bad argument");
  GPRB_REQUIRE(b->inv_ok[gp], "gprb_get_Kinv: the last evaluation was value-only (no inverse resident)");
  std::vector<double> h;
  int rc = fetch_matrix(b, b->A + (size_t)gp * b->npad * b->npad, h);
  if (rc) return rc;
  const size_t dn = (size_t)b->J * NB * NB;
  std::vector<double> dg(dn);
  GPRB_CUDA(cudaMemcpy(dg.data(), b->KinvD + (size_t)gp * dn, sizeof(double) * dn, cudaMemcpyDeviceToHost));
  const int64_t n = b->n, np = b->npad;
  for (int64_t c = 0; c < n; ++c)
    for (int64_t r = c; r < n; ++r) {
      const int64_t ti = r / NB, tj = c / NB, rl = r % NB, cl = c % NB;
      // tile (ti,tj), ti > tj, lives un-transposed at tile position (tj,ti); diagonal tiles in KinvD
      const double v = (ti == tj) ? dg[(size_t)ti * NB * NB + rl + cl * NB] : h[(tj * NB + rl) + (ti * NB + cl) * np];
      out[r + c * n] = out[c + r * n] = v;
    }
  return GPRB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Full posterior covariance and posterior draws (gprb_predict_cov, gprb_sample_posterior) on prediction slot 0.
// The right-hand sides T = L^-1 K* of every 128-column chunk are kept (one [B][npad][PT] block per chunk behind one tensor
// map), computed by gprb_predict's tiled path (predict_tiles) - the GEMV path never materialises T.  The covariance
// tiles of a stream group follow its last FWD_ROW chain on the group's stream.  Leaves Sigma in pc.S and mu in the slot's
// pmu; t0 recorded.
static int postcov_enqueue(gprb_batch* b, int64_t m, const double* Xstar, int64_t xstar_stride, const double* mstar, bool add_noise) {
  gprb_predict_slot& sl = b->ps[0];
  gprb_postcov_ws& w = b->pc;
  const int count = b->B;
  const int64_t npad = b->npad, mpad = (m + NB - 1) / NB * NB;
  const int nchunk = (int)(mpad / NB);
  int rc;
  if ((rc = ensure_dev(&w.T, &w.T_cap, (size_t)nchunk * count * npad * PT)) ||
      (rc = ensure_dev(&w.S, &w.S_cap, (size_t)count * mpad * mpad)) || (rc = ensure_dev(&w.bad, &w.bad_cap, (size_t)count)) ||
      // T of chunk c, GP g is block c * count + g of the map
      (rc = make_tensor_map(&w.tm_T68, w.T, PT, (uint64_t)npad, (uint64_t)nchunk * count, PT, (uint64_t)npad * PT, NB / 2 + 4, KT)) ||
      (rc = predict_stage(b, 0, 0, count, 1, m, Xstar, xstar_stride, mstar, (size_t)count * m)))
    return rc;
  GPRB_CUDA(cudaMemsetAsync(w.bad, 0, sizeof(int32_t) * count, b->stream[0]));
  PostCovArgs pa{sl.pX, b->theta, sl.mask, w.S, w.bad, xstar_stride, b->gemm.nv, b->d, (int)m, (int)mpad, b->kind, 0, count, 0,
                 add_noise ? 1 : 0, w.tm_T68};
  auto cov = [&](const PredictTileArgs& ta, GemmArgs&, int, int g0, int g1, cudaStream_t ss) {
    if (ta.s0 + ta.mc < m) return 0;  // the covariance tiles wait until every chunk of the group's GPs is solved
    pa.g0 = g0;
    if (int rc = launch_post_cov(pa, g1 - g0, ss)) return rc;
    b->ctx->launches++;
    return 0;
  };
  return predict_tiles(b, 0, 0, count, 1, m, xstar_stride, mstar != nullptr, nullptr, w.T, w.tm_T68, true, true, cov);
}

static int postcov_check(gprb_batch* b, int64_t m, const double* Xstar, int64_t xstar_stride) {
  int rc = predict_check(b, 0, 0, b ? b->B : 1, m, Xstar, xstar_stride);
  if (rc) return rc;
  GPRB_REQUIRE(m <= POSTCOV_MAX_M, "gprb_predict_cov / gprb_sample_posterior: m must be <= 8192");
  return 0;
}

// make_posdef! + blocked Cholesky of Sigma_f for `cnt` GPs (list = nullptr: GPs 0 .. cnt-1) on `st`: the left-looking
// schedule of the evaluation pipeline on the per-call workspace (one k_diag_factor launch when m <= 128).
static int postcov_factor(gprb_batch* b, int64_t m, const int32_t* list, int cnt, cudaStream_t st) {
  gprb_postcov_ws& w = b->pc;
  const int64_t mpad = (m + NB - 1) / NB * NB;
  const int Jm = (int)(mpad / NB), nvm = (int)((m + KT - 1) / KT * KT);
  const int64_t ms = mpad * mpad, dstride = (int64_t)Jm * NB * NB;
  int rc;
  GemmArgs ga{w.L, w.DinvT, w.Dinv, w.S, w.L, nullptr, list, ms, dstride, (int)mpad, Jm, 0, GEMM_CHOL_DIAG, nvm};
  ga.fail = w.fail;
  if (Jm > 1) {
    if ((rc = encode_factor_maps(ga, (uint64_t)b->B))) return rc;
    ga.tm_T68 = w.tm_T68;
  }
  DiagArgs da{w.S, w.L, w.Dinv, w.DinvT, w.logdet, w.fail, list, ms, dstride, (int)mpad, Jm, 0, nvm};
  for (int j = 0; j < Jm; ++j) {
    ga.step = j;
    if (j > 0) {  // S(0,0) = Sigma(0,0): k_diag_factor reads block column 0 straight from the workspace
      ga.mode = GEMM_CHOL_DIAG;
      if ((rc = launch_tile_gemm(ga, 1, cnt, st))) return rc;
      b->ctx->launches++;
    }
    da.step = j;
    da.Src = j == 0 ? w.S : nullptr;
    if ((rc = launch_diag_factor(da, cnt, st))) return rc;
    b->ctx->launches++;
    if (j + 1 < Jm) {
      ga.mode = GEMM_CHOL_COL;
      if ((rc = launch_tile_gemm(ga, Jm - 1 - j, cnt, st))) return rc;
      b->ctx->launches++;
    }
  }
  return 0;
}

extern "C" {

int gprb_predict_cov(gprb_batch* b, int64_t m, const double* Xstar, int64_t xstar_stride, const double* mstar, int32_t add_noise,
                     double* mu, double* cov) {
  GPRB_REQUIRE(b && mu && cov, "gprb_predict_cov: NULL argument");
  int rc = postcov_check(b, m, Xstar, xstar_stride);
  if (rc) return rc;
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  gprb_predict_slot& sl = b->ps[0];
  gprb_postcov_ws& w = b->pc;
  const int B = b->B;
  const int64_t mpad = (m + NB - 1) / NB * NB;
  if ((rc = ensure_dev(&w.O, &w.O_cap, (size_t)B * m * m))) return rc;
  if ((rc = postcov_enqueue(b, m, Xstar, xstar_stride, mstar, add_noise != 0))) return rc;
  cudaStream_t st = b->stream[0];
  // pack Sigma [B][mpad][mpad] -> [B][m][m] on the device, so that the copy to the host is one contiguous transfer
  cudaMemcpy3DParms p = {};
  p.srcPtr = make_cudaPitchedPtr(w.S, sizeof(double) * mpad, sizeof(double) * mpad, mpad);
  p.dstPtr = make_cudaPitchedPtr(w.O, sizeof(double) * m, sizeof(double) * m, m);
  p.extent = make_cudaExtent(sizeof(double) * m, m, B);
  p.kind = cudaMemcpyDeviceToDevice;
  GPRB_CUDA(cudaMemcpy3DAsync(&p, st));
  GPRB_CUDA(cudaEventRecord(sl.t1, st));  // device time: the m x m blocks' copy to the host is not part of it
  GPRB_CUDA(cudaMemcpyAsync(sl.h_out, sl.pmu, sizeof(double) * B * m, cudaMemcpyDeviceToHost, st));
  GPRB_CUDA(cudaMemcpyAsync(cov, w.O, sizeof(double) * B * m * m, cudaMemcpyDeviceToHost, st));
  GPRB_CUDA(cudaStreamSynchronize(st));
  if ((rc = slot_wait(sl))) return rc;
  memcpy(mu, sl.h_out, sizeof(double) * B * m);
  return GPRB_OK;
}

int gprb_sample_posterior(gprb_batch* b, int64_t m, const double* Xstar, int64_t xstar_stride, const double* mstar, int32_t ns,
                          const double* Z, double* out, int32_t* info) {
  GPRB_REQUIRE(b && Z && out && info, "gprb_sample_posterior: NULL argument");
  GPRB_REQUIRE(ns >= 1, "gprb_sample_posterior: ns must be >= 1");
  int rc = postcov_check(b, m, Xstar, xstar_stride);
  if (rc) return rc;
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  gprb_predict_slot& sl = b->ps[0];
  gprb_postcov_ws& w = b->pc;
  const int B = b->B;
  const int64_t mpad = (m + NB - 1) / NB * NB, Jm = mpad / NB;
  const size_t nz = (size_t)B * ns * m;
  if ((rc = ensure_dev(&w.L, &w.L_cap, (size_t)B * mpad * mpad)) || (rc = ensure_dev(&w.logdet, &w.logdet_cap, (size_t)B * Jm)) ||
      (rc = ensure_dev(&w.Z, &w.Z_cap, nz)) || (rc = ensure_dev(&w.O, &w.O_cap, nz)) ||
      (rc = ensure_dev(&w.fail, &w.fail_cap, (size_t)B)) || (rc = ensure_dev(&w.list, &w.list_cap, (size_t)B)))
    return rc;
  if (w.D_cap < (size_t)B * Jm * NB * NB) {  // k_diag_factor writes only the triangular halves: the other halves stay zero
    if ((rc = ensure_dev(&w.Dinv, &w.D_cap, (size_t)B * Jm * NB * NB, true))) return rc;
    cudaFree(w.DinvT);
    w.DinvT = nullptr;
    if ((rc = dev_alloc(&w.DinvT, w.D_cap))) { w.D_cap = 0; return rc; }
    GPRB_CUDA(cudaMemset(w.DinvT, 0, sizeof(double) * w.D_cap));
  }
  if (!w.fail_host) {
    GPRB_CUDA(cudaMallocHost((void**)&w.fail_host, sizeof(int32_t) * B));
    GPRB_CUDA(cudaMallocHost((void**)&w.list_host, sizeof(int32_t) * B));
    GPRB_CUDA(cudaEventCreateWithFlags(&w.z_ready, cudaEventDisableTiming));
  }
  if ((rc = postcov_enqueue(b, m, Xstar, xstar_stride, mstar, false))) return rc;
  cudaStream_t st = b->stream[0];
  // the draws' standard normals (m ns B doubles, 32 MB at m = ns = 100, B = 400) travel on the upload stream while the
  // device solves for T; only the draws wait for them
  GPRB_CUDA(cudaMemcpyAsync(w.Z, Z, sizeof(double) * nz, cudaMemcpyHostToDevice, b->ctx->upload));
  GPRB_CUDA(cudaEventRecord(w.z_ready, b->ctx->upload));
  if ((rc = launch_post_fail_init(w.fail, sl.mask, w.bad, 0, B, st))) return rc;
  // make_posdef! ladder, like eval_pass: every attempt factorises the GPs still pending, a failed GP gets one more
  // cumulative jitter and is re-submitted alone, at most MAX_JITTER times
  std::vector<int32_t> tries(B, 0), pend;
  for (int i = 0; i < B; ++i) info[i] = 0;
  const int32_t* list = nullptr;
  int cnt = B;
  for (;;) {
    if ((rc = postcov_factor(b, m, list, cnt, st))) return rc;
    GPRB_CUDA(cudaMemcpyAsync(w.fail_host, w.fail, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    GPRB_CUDA(cudaStreamSynchronize(st));
    std::vector<int32_t> retry;
    for (int k = 0; k < cnt; ++k) {
      const int g = list ? pend[k] : k;
      if (posdef_retry(w.fail_host[g], tries[g], info[g])) retry.push_back(g);
    }
    if (retry.empty()) break;
    pend = retry;
    cnt = (int)pend.size();
    memcpy(w.list_host, pend.data(), sizeof(int32_t) * cnt);
    GPRB_CUDA(cudaMemcpyAsync(w.list, w.list_host, sizeof(int32_t) * cnt, cudaMemcpyHostToDevice, st));
    if ((rc = launch_post_jitter(w.S, w.fail, w.list, (int)m, (int)mpad, cnt, st))) return rc;
    b->ctx->launches++;
    list = w.list;
  }
  GPRB_CUDA(cudaStreamWaitEvent(st, w.z_ready, 0));
  PostDrawArgs da{w.L, sl.pmu, w.Z, w.fail, w.O, (int)m, (int)mpad, ns};
  if ((rc = launch_post_draws(da, B, st))) return rc;
  b->ctx->launches++;
  GPRB_CUDA(cudaEventRecord(sl.t1, st));
  GPRB_CUDA(cudaMemcpyAsync(out, w.O, sizeof(double) * nz, cudaMemcpyDeviceToHost, st));
  GPRB_CUDA(cudaStreamSynchronize(st));
  return slot_wait(sl);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Leave-one-out cross-validation (gprb_eval_loo; kernels in loo.cu).  Value only: one pointwise launch over the batch.
// With the gradient, per group of consecutive GPs: pointwise terms, u = K^-1 (alpha ./ d) by k_solve on the resident
// factor, G = diag(sqrt(-c)) K^-1, W = -G'G (zero-initialised k_post_cov), A' = [K | -Q'], then the fused gradient
// kernels unchanged on A' with a zero alpha.  launch_solve / launch_grad index every buffer by the GP index of their
// launch: the batch buffers are passed offset to the group's first GP, the group buffers as they are.
constexpr size_t LOO_WS_BYTES = (size_t)8 << 30;  // bound of the group buffers (about 2 npad^2 doubles per GP)

static void loo_free_groups(gprb_loo_ws& w) {
  cudaFree(w.M); cudaFree(w.W); cudaFree(w.KD); cudaFree(w.vec); cudaFree(w.part); cudaFree(w.mll);
  w.M = w.W = w.KD = w.vec = w.part = w.mll = nullptr;
  w.cap = 0;
}

// Group buffers for `want` GPs; when the device cannot hold them, for half as many, down to one GP.
static int loo_alloc_groups(gprb_batch* b, int want) {
  gprb_loo_ws& w = b->loo;
  if (w.cap >= want) return 0;
  loo_free_groups(w);
  const size_t mat = (size_t)b->npad * b->npad, dn = (size_t)b->J * NB * NB;
  const size_t part = (size_t)b->J * (b->J + 1) / 2 * GRAD_PARTS_PER_TILE * b->P;
  for (int cap = want;; cap = std::max(1, cap / 2)) {
    int rc;
    if (!(rc = dev_alloc(&w.M, cap * mat)) && !(rc = dev_alloc(&w.W, cap * mat)) && !(rc = dev_alloc(&w.KD, cap * dn)) &&
        !(rc = dev_alloc(&w.vec, 5 * (size_t)cap * b->npad)) && !(rc = dev_alloc(&w.part, cap * part)) &&
        !(rc = dev_alloc(&w.mll, (size_t)cap))) {
      GPRB_CUDA(cudaMemset(w.vec + 4 * (size_t)cap * b->npad, 0, sizeof(double) * cap * b->npad));  // the zero alpha
      w.cap = cap;
      return 0;
    }
    loo_free_groups(w);
    if (rc != GPRB_ERR_NOMEM || cap == 1) return rc;
    cudaGetLastError();  // an allocation failure is not sticky: clear it and try a smaller group
  }
}

static int loo_stage(gprb_batch* b, const uint8_t* mode, const std::vector<int32_t>& info, double* logp, double* grad,
                     double* mu, double* var) {
  gprb_loo_ws& w = b->loo;
  const int B = b->B, P = b->P, J = b->J;
  const int64_t n = b->n, npad = b->npad, ms = npad * npad, ds = (int64_t)J * NB * NB;
  const size_t nout = (size_t)B * (1 + P + 2 * n);
  int rc;
  if ((rc = ensure_dev(&w.out, &w.out_cap, nout))) return rc;
  if (!w.skip) {
    if ((rc = dev_alloc(&w.skip, (size_t)B))) return rc;
    GPRB_CUDA(cudaMallocHost((void**)&w.skip_host, sizeof(int32_t) * B));
  }
  double* d_logp = w.out;
  double* d_grad = d_logp + B;
  double* d_mu = d_grad + (size_t)B * P;
  double* d_var = d_mu + (size_t)B * n;
  bool any = false;
  for (int i = 0; i < B; ++i) {
    w.skip_host[i] = (mode[i] && info[i] >= 0) ? 0 : 1;
    any = any || !w.skip_host[i];
  }
  cudaStream_t st = b->stream[0];
  int64_t& launches = b->ctx->launches;
  if (any) {
    GPRB_CUDA(cudaMemcpyAsync(w.skip, w.skip_host, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
    LooArgs la{b->A, b->KinvD, b->alpha, b->ymm, w.skip, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
               d_mu, d_var, d_logp, ms, ds, (int)n, (int)npad, J, 0};
    if (!grad) {
      if ((rc = launch_loo_point(la, B, st))) return rc;
      ++launches;
    } else {
      const size_t per_gp = sizeof(double) * (2 * (size_t)ms + ds + 5 * npad + (size_t)J * (J + 1) / 2 * GRAD_PARTS_PER_TILE * P + 1);
      if ((rc = loo_alloc_groups(b, (int)std::max<size_t>(1, std::min<size_t>(B, LOO_WS_BYTES / per_gp))))) return rc;
      const int cap = std::min(w.cap, B), nv = (int)((n + KT - 1) / KT * KT);
      double* v = w.vec;
      double* s = v + (size_t)cap * npad;
      double* u = s + (size_t)cap * npad;
      double* z = u + (size_t)cap * npad;
      const double* zero = z + (size_t)cap * npad;
      for (int g0 = 0; g0 < B; g0 += cap) {
        const int cnt = std::min(cap, B - g0);
        bool work = false;
        for (int i = g0; i < g0 + cnt; ++i) work = work || !w.skip_host[i];
        if (!work) continue;
        la.gp0 = g0; la.v = v; la.s = s; la.u = u; la.G = w.M; la.W = w.W; la.Ap = w.M; la.KinvDp = w.KD;
        if ((rc = launch_loo_point(la, cnt, st))) return rc;
        SolveArgs sa{b->Lm + g0 * ms, b->Dinv + g0 * ds, v, b->logdet_part + (int64_t)g0 * J, w.skip + g0, z, u, w.mll, nullptr,
                     ms, ds, (int)n, (int)npad, J, nv};
        sa.cluster_below = b->solve_cluster_below;
        if ((rc = launch_solve(sa, cnt, st))) return rc;
        if ((rc = launch_loo_expand(la, cnt, st))) return rc;
        PostCovArgs pa{nullptr, b->theta + (int64_t)g0 * P, w.skip + g0, w.W, nullptr, 0, nv, b->d, (int)n, (int)npad, b->kind,
                       0, cnt, 0, 0, {}};
        if ((rc = make_tensor_map(&pa.tm_T68, w.M, PT, (uint64_t)npad, (uint64_t)J * cnt, PT, (uint64_t)npad * PT, NB / 2 + 4, KT)))
          return rc;
        if ((rc = launch_loo_w(pa, cnt, st))) return rc;
        if ((rc = launch_loo_assemble(la, cnt, st))) return rc;
        GradArgs gr{b->Xtptr + g0, b->theta + (int64_t)g0 * P, w.M, w.KD, zero, w.part, d_grad + (int64_t)g0 * P, w.skip + g0,
                    nullptr, ms, ds, (int)n, (int)npad, b->d, J, b->kind};
        if ((rc = launch_grad(gr, cnt, st))) return rc;
        launches += 7;  // point, solve, expand, W, assemble, gradient tiles + reduction
      }
    }
  }
  std::vector<double> h(nout);
  if (any) {
    GPRB_CUDA(cudaMemcpyAsync(h.data(), d_logp, sizeof(double) * B, cudaMemcpyDeviceToHost, st));
    if (grad) GPRB_CUDA(cudaMemcpyAsync(h.data() + B, d_grad, sizeof(double) * B * P, cudaMemcpyDeviceToHost, st));
    if (mu || var) GPRB_CUDA(cudaMemcpyAsync(h.data() + B + (size_t)B * P, d_mu, sizeof(double) * 2 * B * n, cudaMemcpyDeviceToHost, st));
    GPRB_CUDA(cudaStreamSynchronize(st));
  }
  const double ninf = -std::numeric_limits<double>::infinity(), qnan = std::numeric_limits<double>::quiet_NaN();
  const double* hg = h.data() + B;
  const double* hm = hg + (size_t)B * P;
  const double* hv = hm + (size_t)B * n;
  for (int gp = 0; gp < B; ++gp) {
    if (!mode[gp]) continue;
    const bool ok = info[gp] >= 0;
    logp[gp] = ok ? h[gp] : ninf;
    if (grad)
      for (int p = 0; p < P; ++p) grad[(size_t)gp * P + p] = ok ? hg[(size_t)gp * P + p] : qnan;
    for (int64_t i = 0; i < n; ++i) {
      if (mu) mu[(size_t)gp * n + i] = ok ? hm[(size_t)gp * n + i] : qnan;
      if (var) var[(size_t)gp * n + i] = ok ? hv[(size_t)gp * n + i] : qnan;
    }
  }
  return 0;
}

extern "C" {

int gprb_eval_loo(gprb_batch* b, const double* theta, const uint8_t* active, double* mll, double* grad, double* logp_loo,
                  double* grad_loo, double* mu_loo, double* var_loo, int32_t* info) {
  GPRB_REQUIRE(b && theta && logp_loo && info, "gprb_eval_loo: NULL argument");
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  const int B = b->B;
  // the evaluation of gprb_eval with a gradient (the LOO terms need K^-1), with its state reuse
  std::vector<uint8_t> mode(B);
  std::vector<int32_t> act;
  for (int i = 0; i < B; ++i) {
    mode[i] = (!active || active[i]) ? 2 : 0;
    if (mode[i]) act.push_back(i);
  }
  int rc = upload_theta_rows(b, theta, act);
  if (rc) return rc;
  std::vector<int32_t> inf;
  if ((rc = evaluate_modes(b, theta, mode.data(), inf))) return rc;
  std::vector<double> tmll, tgrad;
  if (!mll) { tmll.resize(B); mll = tmll.data(); }
  if (!grad) { tgrad.resize((size_t)B * b->P); grad = tgrad.data(); }
  if ((rc = download_results(b, mode.data(), inf, nullptr, mll, grad, info))) return rc;
  return loo_stage(b, mode.data(), inf, logp_loo, grad_loo, mu_loo, var_loo);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Predictive gradients (gprb_predict_grad) on prediction slot 0, chunk by chunk (128 test columns): gprb_predict's tiled
// path (predict_tiles; the FWD_ROW chain T = L^-1 K* only when a variance is asked for), where each stream group then
// runs k_predict_finish for its own mu / var (the launches gprb_predict issues, so mu and var are bit-identical to it),
// the BWD_ROW chain (beta = L^-T T in place, only with dvar) and k_predict_jac.
static int predgrad_enqueue(gprb_batch* b, int64_t m, const double* Xstar, int64_t xstar_stride, const double* mstar,
                            const double* dmstar, bool want_var, bool want_dvar) {
  gprb_predict_slot& sl = b->ps[0];
  gprb_predgrad_ws& w = b->pg;
  const int J = b->J, count = b->B, d = b->d;
  const int64_t npad = b->npad;
  cudaStream_t st = b->stream[0];
  const bool want_T = want_var || want_dvar;
  const size_t nout = (size_t)count * m, njac = nout * d;
  int rc;
  if ((rc = ensure_dev(&w.jac, &w.jac_cap, (want_dvar ? 2 : 1) * njac))) return rc;
  if (dmstar && (rc = ensure_dev(&w.dms, &w.dms_cap, njac))) return rc;
  if (want_var && (rc = ensure_dev(&sl.pvar, &sl.pvar_cap, nout))) return rc;
  if (want_T && (rc = slot_rhs(b, sl, count))) return rc;
  if ((rc = predict_stage(b, 0, 0, count, 1, m, Xstar, xstar_stride, mstar, 2 * nout))) return rc;
  if (dmstar) GPRB_CUDA(cudaMemcpyAsync(w.dms, dmstar, sizeof(double) * njac, cudaMemcpyHostToDevice, st));
  auto jac = [&](const PredictTileArgs& ta, GemmArgs& ga, int ntl, int g0, int g1, cudaStream_t ss) {
    // the group's mu / var: k_predict_finish indexes its outputs and T by blockIdx, so the group's GPs start at g0
    PredictTileArgs tg = ta;
    tg.gp_off = g0;
    if (tg.T) tg.T += (size_t)g0 * npad * PT;
    tg.mupart += (size_t)g0 * J * PT;
    tg.mu += (size_t)g0 * m;
    if (tg.var) tg.var += (size_t)g0 * m;
    if (tg.mstar) tg.mstar += (size_t)g0 * m;
    int rc;
    if ((rc = launch_predict_finish(tg, g1 - g0, ss))) return rc;
    b->ctx->launches++;
    if (want_dvar && (rc = row_chain(b, ga, GEMM_BWD_ROW, ntl, g1 - g0, ss))) return rc;
    PredictJacArgs ja{b->Xtptr, b->theta, b->alpha, want_dvar ? sl.pT + (size_t)g0 * npad * PT : nullptr,
                      sl.pX + (size_t)g0 * xstar_stride, dmstar ? w.dms + (size_t)g0 * m * d : nullptr,
                      w.jac + (size_t)g0 * m * d, want_dvar ? w.jac + njac + (size_t)g0 * m * d : nullptr, sl.mask,
                      xstar_stride, (int)b->n, (int)npad, d, (int)m, b->kind, ta.s0, ta.mc, g0};
    if ((rc = launch_predict_jac(ja, g1 - g0, ss))) return rc;
    b->ctx->launches++;
    return 0;
  };
  if ((rc = predict_tiles(b, 0, 0, count, 1, m, xstar_stride, mstar != nullptr, want_var ? sl.pvar : nullptr,
                          want_T ? sl.pT : nullptr, sl.tm_T68, false, false, jac)))
    return rc;
  GPRB_CUDA(cudaMemcpyAsync(sl.h_out, sl.pmu, sizeof(double) * nout, cudaMemcpyDeviceToHost, st));
  if (want_var) GPRB_CUDA(cudaMemcpyAsync(sl.h_out + nout, sl.pvar, sizeof(double) * nout, cudaMemcpyDeviceToHost, st));
  GPRB_CUDA(cudaEventRecord(sl.t1, st));
  return 0;
}

extern "C" {

int gprb_predict_grad(gprb_batch* b, int64_t m, const double* Xstar, int64_t xstar_stride, const double* mstar,
                      const double* dmstar, double* mu, double* var, double* dmu, double* dvar) {
  GPRB_REQUIRE(b && mu && dmu, "gprb_predict_grad: NULL argument");
  int rc = predict_check(b, 0, 0, b->B, m, Xstar, xstar_stride);
  if (rc) return rc;
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  if ((rc = predgrad_enqueue(b, m, Xstar, xstar_stride, mstar, dmstar, var != nullptr, dvar != nullptr))) return rc;
  gprb_predict_slot& sl = b->ps[0];
  cudaStream_t st = b->stream[0];
  const size_t nout = (size_t)b->B * m, njac = nout * b->d;
  // the Jacobians go straight to the caller's memory, after t1: the device time does not include their copy
  GPRB_CUDA(cudaMemcpyAsync(dmu, b->pg.jac, sizeof(double) * njac, cudaMemcpyDeviceToHost, st));
  if (dvar) GPRB_CUDA(cudaMemcpyAsync(dvar, b->pg.jac + njac, sizeof(double) * njac, cudaMemcpyDeviceToHost, st));
  GPRB_CUDA(cudaStreamSynchronize(st));
  if ((rc = slot_wait(sl))) return rc;
  memcpy(mu, sl.h_out, sizeof(double) * nout);
  if (var) memcpy(var, sl.h_out + nout, sizeof(double) * nout);
  return GPRB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Appending samples (gprb_batch_append; GaussianProcesses ElasticGPE append!).  The left-looking factorisation computes
// the tiles of block row i from K's block rows i and j and from L(., k < j) only, and the assembly centres at the
// dataset's first sample: with j0 = floor(n_old / 128), the block rows < j0 of K, L, the inverted diagonal blocks and the
// logdet partials on n_old + k samples are bit for bit the resident ones.  The incremental pass (enqueue_pipeline with j0)
// recomputes the rest, so a GP ends in exactly the state gprb_eval(theta, value only) leaves on the enlarged data.

// The leading rows x cols of every GP's column-major block, from leading dimension lds (blocks of lds x scols) to ldd
// (blocks of ldd x dcols), all GPs in one 3-D copy.
static int restride(double* dst, int64_t ldd, int64_t dcols, const double* src, int64_t lds, int64_t scols, int64_t rows,
                    int64_t cols, int B, cudaStream_t st) {
  cudaMemcpy3DParms p = {};
  p.srcPtr = make_cudaPitchedPtr(const_cast<double*>(src), sizeof(double) * lds, sizeof(double) * lds, scols);
  p.dstPtr = make_cudaPitchedPtr(dst, sizeof(double) * ldd, sizeof(double) * ldd, dcols);
  p.extent = make_cudaExtent(sizeof(double) * rows, cols, B);
  p.kind = cudaMemcpyDeviceToDevice;
  GPRB_CUDA(cudaMemcpy3DAsync(&p, st));
  return 0;
}

// Move one [B][ld][ld] matrix to a new allocation of leading dimension ld1, keeping its leading keep x keep block; the
// old allocation is freed only after the copy, so a failed allocation leaves *p as it was.
static int move_matrix(gprb_batch* b, double** p, int64_t ld0, int64_t ld1, int64_t keep) {
  double* q = nullptr;
  int rc = dev_alloc(&q, (size_t)b->B * ld1 * ld1);
  if (rc) return rc;
  if (!(rc = restride(q, ld1, ld1, *p, ld0, ld0, keep, keep, b->B, b->stream[0]))) {
    cudaError_t e = cudaStreamSynchronize(b->stream[0]);
    if (e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize(move_matrix)", __FILE__, __LINE__);
  }
  if (rc) { cudaFree(q); return rc; }
  cudaFree(*p);
  *p = q;
  return 0;
}

// The [B][npad] / [B][J] buffers of a batch at a new npad, J (allocated all or none).
struct GrownBuffers {
  double *Dinv = nullptr, *DinvT = nullptr, *KinvD = nullptr, *logdet = nullptr, *gpart = nullptr, *ymm = nullptr,
         *alpha = nullptr, *zbuf = nullptr;
  void release() {
    for (double* p : {Dinv, DinvT, KinvD, logdet, gpart, ymm, alpha, zbuf}) cudaFree(p);
    *this = GrownBuffers{};
  }
};

static int grow_alloc(gprb_batch* b, GrownBuffers& g, int64_t np1, int J1) {
  const size_t B = (size_t)b->B, dinv = (size_t)J1 * NB * NB, ntiles = (size_t)J1 * (J1 + 1) / 2;
  int rc;
  if ((rc = dev_alloc(&g.Dinv, dinv * B)) || (rc = dev_alloc(&g.DinvT, dinv * B)) || (rc = dev_alloc(&g.KinvD, dinv * B)) ||
      (rc = dev_alloc(&g.logdet, B * J1)) || (rc = dev_alloc(&g.gpart, B * ntiles * GRAD_PARTS_PER_TILE * b->P)) ||
      (rc = dev_alloc(&g.ymm, B * np1)) || (rc = dev_alloc(&g.alpha, B * np1)) || (rc = dev_alloc(&g.zbuf, B * np1)))
    g.release();
  return rc;
}

// Grow-only workspaces whose shape or tensor maps derive from npad or J: released, the next call allocates them again.
// (gprb_predgrad_ws is sized by m and d only.)
static void release_npad_workspaces(gprb_batch* b) {
  for (gprb_predict_slot& sl : b->ps) {
    cudaFree(sl.pT); sl.pT = nullptr; sl.pT_cap = 0; sl.tm_T_cap = 0;
    cudaFree(sl.pmupart); sl.pmupart = nullptr; sl.pmupart_cap = 0;
  }
  cudaFree(b->pc.T); b->pc.T = nullptr; b->pc.T_cap = 0;
  loo_free_groups(b->loo);
}

extern "C" {

int gprb_batch_append(gprb_batch* b, int64_t k, const double* const* Xnew, int64_t ldx, const double* ymm_new, double* mll,
                      int32_t* info) {
  GPRB_REQUIRE(b && Xnew && ymm_new, "gprb_batch_append: NULL argument");
  GPRB_REQUIRE(k >= 1, "gprb_batch_append: k must be >= 1");
  GPRB_REQUIRE(ldx >= b->d, "gprb_batch_append: ldx < d");
  GPRB_REQUIRE(b->n + k <= (1 << 20), "gprb_batch_append: n + k out of range");
  GPRB_REQUIRE(!b->ps[0].pending && !b->ps[1].pending,
               "gprb_batch_append: a prediction is in flight - call gprb_predict_wait first");
  const std::vector<gprb_dataset*> uds = distinct_datasets(b);
  const int T = (int)uds.size();
  for (int t = 0; t < T; ++t) {
    GPRB_REQUIRE(Xnew[t] != nullptr, "gprb_batch_append: NULL input block");
    GPRB_REQUIRE(uds[t]->users == 1, "gprb_batch_append: a dataset of the batch is also used by another live batch");
  }
  GPRB_CUDA(cudaSetDevice(b->ctx->device));
  const int B = b->B, P = b->P, d = b->d;
  cudaStream_t st = b->stream[0];
  const int64_t n0 = b->n, np0 = b->npad, n1 = n0 + k, np1 = (n1 + NB - 1) / NB * NB;
  const int J0 = b->J, J1 = (int)(np1 / NB), j0 = (int)(n0 / NB);
  if ((int)b->theta_valid.size() != B) {
    b->theta_valid.assign(B, 0); b->theta_last.assign((size_t)B * P, 0.0); b->info_last.assign(B, 0); b->ds_ver.assign(B, 0);
  }
  // theta of every resident state (gprb_eval_device states included: the device copy is the one that was evaluated)
  std::vector<double> theta((size_t)B * P);
  GPRB_CUDA(cudaStreamSynchronize(st));
  GPRB_CUDA(cudaMemcpy(theta.data(), b->theta, sizeof(double) * B * P, cudaMemcpyDeviceToHost));
  // incremental: a state factorised without jitter (the jitter 1e-6 tr(K)/n changes with n) that keeps whole block rows
  std::vector<uint8_t> mode(B, 0);
  std::vector<int32_t> inc, fall;
  for (int i = 0; i < B; ++i) {
    if (!b->state_ok[i]) continue;
    mode[i] = 1;
    (b->info_last[i] == 0 && j0 >= 1 ? inc : fall).push_back(i);
  }

  // ---- device memory: every allocation before anything is freed or overwritten
  gprb_slab* sl = new (std::nothrow) gprb_slab();
  GPRB_REQUIRE(sl != nullptr, "gprb_batch_append: out of host memory");
  int rc;
  if ((rc = dev_alloc(&sl->X, (size_t)T * d * n1)) || (rc = dev_alloc(&sl->Xt, (size_t)T * d * np1))) {
    cudaFree(sl->X); cudaFree(sl->Xt); delete sl;
    return rc;
  }
  if (np1 > np0) {
    release_npad_workspaces(b);
    GrownBuffers g;
    // one large matrix at a time: the peak is the resident buffers plus one new [B][npad][npad] copy
    if ((rc = grow_alloc(b, g, np1, J1)) || (rc = move_matrix(b, &b->A, np0, np1, np0))) {
      g.release(); cudaFree(sl->X); cudaFree(sl->Xt); delete sl;
      return rc;
    }
    if ((rc = move_matrix(b, &b->Lm, np0, np1, np0))) {
      if (move_matrix(b, &b->A, np1, np0, np0) == 0) set_batch_gemm(b);  // back to the old stride (its memory was just freed)
      else set_error("gprb_batch_append: out of device memory, and the batch could not be restored");
      g.release(); cudaFree(sl->X); cudaFree(sl->Xt); delete sl;
      return rc;
    }
    const size_t dn0 = (size_t)J0 * NB * NB, dn1 = (size_t)J1 * NB * NB;
    // k_diag_factor writes only the triangular halves of the inverted diagonal blocks: the other halves stay zero
    GPRB_CUDA(cudaMemsetAsync(g.Dinv, 0, sizeof(double) * dn1 * B, st));
    GPRB_CUDA(cudaMemsetAsync(g.DinvT, 0, sizeof(double) * dn1 * B, st));
    GPRB_CUDA(cudaMemsetAsync(g.ymm, 0, sizeof(double) * np1 * B, st));  // zero padding
    GPRB_CUDA(cudaMemcpy2DAsync(g.Dinv, sizeof(double) * dn1, b->Dinv, sizeof(double) * dn0, sizeof(double) * dn0, B,
                                cudaMemcpyDeviceToDevice, st));
    GPRB_CUDA(cudaMemcpy2DAsync(g.DinvT, sizeof(double) * dn1, b->DinvT, sizeof(double) * dn0, sizeof(double) * dn0, B,
                                cudaMemcpyDeviceToDevice, st));
    GPRB_CUDA(cudaMemcpy2DAsync(g.logdet, sizeof(double) * J1, b->logdet_part, sizeof(double) * J0, sizeof(double) * J0, B,
                                cudaMemcpyDeviceToDevice, st));
    GPRB_CUDA(cudaMemcpy2DAsync(g.ymm, sizeof(double) * np1, b->ymm, sizeof(double) * np0, sizeof(double) * n0, B,
                                cudaMemcpyDeviceToDevice, st));
    GPRB_CUDA(cudaStreamSynchronize(st));
    for (double* p : {b->Dinv, b->DinvT, b->KinvD, b->logdet_part, b->grad_part, b->ymm, b->alpha, b->zbuf}) cudaFree(p);
    b->Dinv = g.Dinv; b->DinvT = g.DinvT; b->KinvD = g.KinvD; b->logdet_part = g.logdet; b->grad_part = g.gpart;
    b->ymm = g.ymm; b->alpha = g.alpha; b->zbuf = g.zbuf;
  }

  // ---- the grown data: old samples, then the new ones, into the new slab; y - m(X) of the new samples
  for (int t = 0; t < T; ++t) {
    double* x = sl->X + (size_t)t * d * n1;
    GPRB_CUDA(cudaMemcpyAsync(x, uds[t]->X, sizeof(double) * d * n0, cudaMemcpyDeviceToDevice, st));
    GPRB_CUDA(cudaMemcpy2DAsync(x + (size_t)d * n0, sizeof(double) * d, Xnew[t], sizeof(double) * ldx, sizeof(double) * d, k,
                                cudaMemcpyHostToDevice, st));
  }
  if ((rc = launch_transpose_inputs_batched(sl->X, sl->Xt, (int)n1, (int)np1, d, T, st))) return rc;
  b->ctx->launches++;
  GPRB_CUDA(cudaMemcpy2DAsync(b->ymm + n0, sizeof(double) * np1, ymm_new, sizeof(double) * k, sizeof(double) * k, B,
                              cudaMemcpyHostToDevice, st));
  GPRB_CUDA(cudaStreamSynchronize(st));
  sl->count = T; sl->refs = T;
  for (int t = 0; t < T; ++t) {
    gprb_dataset* ds = uds[t];
    if (ds->slab) {
      if (--ds->slab->refs == 0) { cudaFree(ds->slab->X); cudaFree(ds->slab->Xt); delete ds->slab; }
    } else {
      cudaFree(ds->X); cudaFree(ds->Xt);
    }
    ds->n = n1; ds->npad = np1;
    ds->X = sl->X + (size_t)t * d * n1;
    ds->Xt = sl->Xt + (size_t)t * d * np1;
    ds->slab = sl; ds->slab_index = t;
    ds->version++;
  }
  {
    std::vector<const double*> xp(B), xtp(B);
    for (int i = 0; i < B; ++i) { xp[i] = b->ds[i]->X; xtp[i] = b->ds[i]->Xt; }
    GPRB_CUDA(cudaMemcpy(b->Xptr, xp.data(), sizeof(double*) * B, cudaMemcpyHostToDevice));
    GPRB_CUDA(cudaMemcpy(b->Xtptr, xtp.data(), sizeof(double*) * B, cudaMemcpyHostToDevice));
  }
  b->n = n1; b->npad = np1; b->J = J1;
  if ((rc = set_batch_gemm(b))) return rc;
  std::fill(b->inv_ok.begin(), b->inv_ok.end(), (uint8_t)0);
  std::fill(b->v_ok.begin(), b->v_ok.end(), (uint8_t)0);

  // ---- incremental pass over the stream groups; a GP whose new diagonal blocks fail a pivot joins the fallback
  std::vector<int32_t> inf(B, 0);
  if (!inc.empty()) {
    std::vector<Group> groups = build_groups(b, {}, {}, inc);
    for (Group& g : groups) { g.rl = false; g.j0 = j0; }
    GPRB_CUDA(cudaMemcpyAsync(b->list, b->list_host, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
    if ((rc = run_pipeline(b, groups))) return rc;
    GPRB_CUDA(cudaMemcpyAsync(b->fail_host, b->fail, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    GPRB_CUDA(cudaStreamSynchronize(st));
    for (int gp : inc) {
      if (b->fail_host[gp] != 0) { fall.push_back(gp); continue; }
      memcpy(b->theta_last.data() + (size_t)gp * P, theta.data() + (size_t)gp * P, sizeof(double) * P);
      b->theta_valid[gp] = 1; b->info_last[gp] = 0; b->ds_ver[gp] = b->ds[gp]->version;
    }
  }
  // ---- fallback: an ordinary value-only evaluation with the whole make_posdef! ladder at the resident theta
  if (!fall.empty()) {
    std::vector<uint8_t> fm(B, 0);
    for (int gp : fall) fm[gp] = 1;
    std::vector<int32_t> finf;
    if ((rc = evaluate_modes(b, theta.data(), fm.data(), finf))) return rc;
    for (int gp : fall) inf[gp] = finf[gp];
  }
  std::vector<double> tmll;
  std::vector<int32_t> tinfo;
  if (!mll) { tmll.resize(B); mll = tmll.data(); }
  if (!info) { tinfo.resize(B); info = tinfo.data(); }
  return download_results(b, mode.data(), inf, nullptr, mll, nullptr, info);
}

}  // extern "C"
