// Batched fp64 tile GEMM (NT form) on the DMMA tensor pipe - the engine of the blocked
// Cholesky (row a6), the triangular inverse and the LAUUM product (row a8) of SURVEY.md section 8a, and of the
// blocked forward substitution of the predictive variance (row a11).
//
// One CTA = one HALF of a 128x128 output tile of one GP, two CTAs per SM:
//     acc = sum_{k-blocks} Aop[i-rows, k] * Bop[j-rows, k]^T          (both operands column-major, ld = npad)
//   ROWSPLIT kernel (64 rows x 128 columns per CTA): CHOL_DIAG, CHOL_COL, CHOL_PANEL, CHOL_TRAIL, LAUUM
//            - the modes whose post-multiply contracts over the tile's COLUMNS (T * inv(L_jj)^T) or that have none
//   COLSPLIT kernel (128 rows x 64 columns per CTA): TRTRI_ROW, FWD_ROW
//            - the modes whose post-multiply contracts over the tile's ROWS (-inv(L_ii) * T)
// Why halves: a 128x128 fp64 tile pins 203 KB of shared memory, so one CTA owned an SM and every per-tile phase that
// is not the k-loop (pipeline fill 2-8 us, parking the tile for the post-multiply 1-3 us, the store 1-2 us) left the
// DMMA pipe idle - 8-17 us per tile against k-loops of 16.6 us per 128-block (profiles/r01_gemm_tile_timeline.log).
// Half tiles need 108 KB: two CTAs share an SM and the fill / park / store of one runs under the k-loop of the
// other.  Launches with fewer tiles than SMs (the serial CHOL_DIAG chain, small batches, the reference's one-GP-at-
// a-time pattern) get twice the CTAs.
//
// Eight DMMA consumer warps with 32x32 register tiles (mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4, the native fp64 tensor
// shape on sm_100a; tcgen05 has no f64 kind), two per SMSP, and NO producer warp: a whole operand chunk arrives with
// ONE tensor-map TMA request (cp.async.bulk.tensor.3d, SASS UTMALDG; completion counted on mbarriers), so the two
// requests of a chunk are issued by lane 0 of consumer warp 0 right after the stage they refill has been released by
// all eight warps.  256 threads x 2 CTAs leave 128 registers per thread: accumulators (64) plus A/B fragments
// double-buffered a k4-step ahead fit without spills.  Measured steps of this design at B = 400 GPs, n = 2000:
// full tiles + producer warp (round 1) 119.1 ms, half tiles with four 64x32 consumer warps 119.5 ms (a lone warp per
// SMSP leaves bubbles at every chunk boundary, and co-resident CTAs of one launch run in lockstep), eight 32x32 warps
// 115.1 ms.
// Padded smem rows (132 / 68 doubles, both = 4 mod 16) make every fragment load bank-conflict free.
//
// Modes (tile coordinates and k-range derive from `mode`, `step` and blockIdx.x):
//   CHOL_DIAG  S(j,j)   = K(j,j) - sum_{k<j} L(j,k) L(j,k)^T                      -> Lm(j,j)   (potf2 follows)
//   CHOL_COL   L(i,j)   = [K(i,j) - sum_{k<j} L(i,k) L(j,k)^T] * inv(L_jj)^T      -> Lm(i,j)   i > j = step, i >= row0
//   TRTRI_ROW  W(i,j)   = -inv(L_ii) * sum_{k=j}^{i-1} L(i,k) W(k,j)   stored as V(j,i) = W(i,j)^T, i = step
//   LAUUM      Kinv(i,j) = sum_{k>=i} V(i,k) V(j,k)^T  (i >= j)  -> upper tile (j,i) of A (un-transposed) / KinvD(i)
//   CHOL_PANEL L(i,j)   = S(i,j) * inv(L_jj)^T                       in place in Lm, i > j = step      } right-looking
//   CHOL_TRAIL S(i,k)  -= L(i,j) L(k,j)^T   for all j < k <= i          in place in Lm, j = step          } variant
//              (small batches: 3 short launches per block column instead of serial k-loops that grow with the column
//               index)
//   FWD_ROW    T(i,:)   = inv(L_ii) * [T(i,:) - sum_{k<i} L(i,k) T(k,:)]   in place in the right-hand-side block
//              (blocked forward substitution L^-1 K* of the predictive variance, PDMats whiten!), i = step
//   BWD_ROW    B(i,:)   = inv(L_ii)^T [T(i,:) - sum_{k>i} L(k,i)^T B(k,:)]   in place, i = step = J-1 .. 0
//              (blocked backward substitution L^-T (L^-1 K*) of the predictive gradient; its own kernel, k_tile_bwd: the
//               A operand is L's lower tiles read transposed through tm_LT, the post-multiplier inv(L_ii)^T comes from DinvT)
// where V = L^-T lives in the strictly-upper tiles of Lm and its diagonal blocks in DinvT.
// The per-element summation order is that of the full-tile kernel of round 1 (k-blocks ascending, 4 k per DMMA), so
// results are unchanged bit for bit and both Cholesky schedules stay bit-identical to each other.
#include "common.cuh"
#include "kernels.h"

namespace gprb {

// Debug timeline (build with -DGPRB_TIMELINE): warp 0 lane 0 of every tile records globaltimer at phase boundaries.
#ifdef GPRB_TIMELINE
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define GPRB_TL(k) do { if (g.tl && threadIdx.x == 0) g.tl[((int64_t)blockIdx.y * gridDim.x + blockIdx.x) * 8 + (k)] = gtimer(); } while (0)
#else
#define GPRB_TL(k) do { } while (0)
#endif

constexpr int HB = NB / 2;                               // 64: the short edge of a half tile
constexpr int LDS_H = HB + 4;                            // padded smem row of a 64-wide operand chunk (68 = 4 mod 16)
constexpr int NSTAGE = 3;
constexpr int STAGE_DOUBLES = KT * (LDS_T + LDS_H);      // A + B operand chunk (one is 128 wide, the other 64)
constexpr int RBUF_DOUBLES = KT * LDS_T;                 // one chunk of the post-multiplier (always 128 wide)
constexpr int NRBUF = 2;                                 // ring depth of the post-multiplier chunks
constexpr int N_CONSUMER_WARPS = 8;
constexpr int MI_N = 4;                                  // 8-row slabs of a warp tile: 32 x 32 register tiles
constexpr int WROWS = MI_N * 8;                          // rows of a warp tile
constexpr int GEMM_THREADS = N_CONSUMER_WARPS * 32;      // no producer warp: warp 0 issues the (two) TMA requests of a chunk
static_assert(2 * NSTAGE + 2 * NRBUF <= 16, "barrier block holds 16 mbarriers");
static_assert(NSTAGE * STAGE_DOUBLES >= NB * LDS_H, "the parked half tile must fit the stage ring");
constexpr size_t GEMM_SMEM = (size_t)(NSTAGE * STAGE_DOUBLES + NRBUF * RBUF_DOUBLES) * sizeof(double) + 16 * sizeof(uint64_t);
static_assert(2 * (GEMM_SMEM + 1024) <= 228 * 1024, "two CTAs per SM");

struct TileCoord {
  int i, j;        // output tile (block row, block col)
  int kb0, kb1;    // k-block range [kb0, kb1)
  int a_diag_kb;   // k-block whose A operand comes from DinvT (-1: none)
  int b_diag_kb;   // same for B
  int post;        // 0 none, 1 right-multiply by Dinv[rblk]^T, 2 left-multiply by -Dinv[rblk]
  int rblk;
  bool use_cin;    // T = Cin - acc, else T = acc
};

__device__ __forceinline__ void lower_index(int bx, int& i, int& j) {
  i = (int)((__fsqrt_rn(8.0f * bx + 1.0f) - 1.0f) * 0.5f);  // approximate, corrected by the two loops below
  while ((i + 1) * (i + 2) / 2 <= bx) ++i;
  while (i * (i + 1) / 2 > bx) --i;
  j = bx - i * (i + 1) / 2;
}

__device__ __forceinline__ TileCoord tile_coord(int mode, int step, int J, int row0, int bx) {
  TileCoord tc;
  tc.a_diag_kb = tc.b_diag_kb = -1;
  tc.post = 0;
  tc.rblk = 0;
  tc.use_cin = false;
  if (mode == GEMM_CHOL_DIAG) {
    tc.i = tc.j = step; tc.kb0 = 0; tc.kb1 = step; tc.use_cin = true;
  } else if (mode == GEMM_CHOL_COL) {
    tc.i = max(step + 1, row0) + bx; tc.j = step; tc.kb0 = 0; tc.kb1 = step; tc.use_cin = true; tc.post = 1; tc.rblk = step;
  } else if (mode == GEMM_TRTRI_ROW) {
    tc.i = step; tc.j = bx; tc.kb0 = bx; tc.kb1 = step; tc.b_diag_kb = bx; tc.post = 2; tc.rblk = step;
  } else if (mode == GEMM_CHOL_PANEL) {
    tc.i = step + 1 + bx; tc.j = step; tc.kb0 = 0; tc.kb1 = 0; tc.use_cin = true; tc.post = 1; tc.rblk = step;
  } else if (mode == GEMM_CHOL_TRAIL) {  // bx enumerates the lower tiles of the trailing submatrix, row by row
    int ii, jj;
    lower_index(bx, ii, jj);
    tc.i = step + 1 + ii; tc.j = step + 1 + jj; tc.kb0 = step; tc.kb1 = step + 1; tc.use_cin = true;
  } else if (mode == GEMM_FWD_ROW) {
    tc.i = step; tc.j = bx; tc.kb0 = 0; tc.kb1 = step; tc.use_cin = true; tc.post = 2; tc.rblk = step;
  } else {  // GEMM_LAUUM: bx enumerates (i, j), j <= i, row by row => longest k-range first
    int i, j;
    lower_index(bx, i, j);
    tc.i = i; tc.j = j; tc.kb0 = i; tc.kb1 = J; tc.a_diag_kb = i;
    tc.b_diag_kb = (j == i) ? i : -1;
  }
  return tc;
}

enum { SEL_FULL = 0, SEL_SKIP, SEL_MI2, SEL_NI1, SEL_NI2, SEL_NI3, SEL_TRI0, SEL_MLO2, SEL_MLO2_NI3, SEL_NLO2 };

// One k-chunk (KT = 16) of a warp's 64x32 register tile restricted, at compile time, to the 8x8 blocks
// (mi, ni) with MI_LO <= mi < MI_LIM, NI_LO <= ni < NI_LIM and mi >= ni + OFF: straight-line unpredicated DMMAs.
// LDA / LDB: smem row strides of the two k-major operand chunks.  AK / AM: k and row strides of the A operand (k-major:
// LDA and 1; the row-major A chunk of BWD_ROW: 1 and KT).
template <int LDA, int LDB, int MI_LIM, int NI_LIM, int OFF, int MI_LO = 0, int NI_LO = 0, int AK = LDA, int AM = 1>
__device__ __forceinline__ void chunk_mma(double (&acc)[MI_N][4][2], const double* ap, const double* bp) {
  // ap / bp: this lane's fragment pointers at k4 = 0, i.e. base + t * LD + row0 (resp. col0)
#pragma unroll
  for (int k4 = 0; k4 < KT / 4; ++k4, ap += 4 * AK, bp += 4 * LDB) {
    double a[MI_N], b[4];
#pragma unroll
    for (int mi = MI_LO; mi < MI_LIM; ++mi)
      if (mi >= OFF) a[mi] = ap[mi * 8 * AM];
#pragma unroll
    for (int ni = NI_LO; ni < NI_LIM; ++ni)
      if (ni + OFF <= MI_N - 1) b[ni] = bp[ni * 8];
#pragma unroll
    for (int mi = MI_LO; mi < MI_LIM; ++mi)
#pragma unroll
      for (int ni = NI_LO; ni < NI_LIM; ++ni)
        if (mi >= ni + OFF) dmma884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
  }
}

// Dispatch one chunk to the specialised body `sel` (warp-uniform).
template <int LDA, int LDB, int AK = LDA, int AM = 1>
__device__ __forceinline__ void chunk_dispatch(int sel, double (&acc)[MI_N][4][2], const double* ap, const double* bp) {
  switch (sel) {
    case SEL_SKIP: break;
    case SEL_MI2: chunk_mma<LDA, LDB, 2, 4, -64, 0, 0, AK, AM>(acc, ap, bp); break;
    case SEL_NI1: chunk_mma<LDA, LDB, MI_N, 1, -64, 0, 0, AK, AM>(acc, ap, bp); break;
    case SEL_NI2: chunk_mma<LDA, LDB, MI_N, 2, -64, 0, 0, AK, AM>(acc, ap, bp); break;
    case SEL_NI3: chunk_mma<LDA, LDB, MI_N, 3, -64, 0, 0, AK, AM>(acc, ap, bp); break;
    case SEL_TRI0: chunk_mma<LDA, LDB, MI_N, 4, 0, 0, 0, AK, AM>(acc, ap, bp); break;
    case SEL_MLO2: chunk_mma<LDA, LDB, MI_N, 4, -64, 2, 0, AK, AM>(acc, ap, bp); break;
    case SEL_MLO2_NI3: chunk_mma<LDA, LDB, MI_N, 3, -64, 2, 0, AK, AM>(acc, ap, bp); break;
    case SEL_NLO2: chunk_mma<LDA, LDB, MI_N, 4, -64, 0, 2, AK, AM>(acc, ap, bp); break;
    default: chunk_mma<LDA, LDB, MI_N, 4, -64, 0, 0, AK, AM>(acc, ap, bp); break;
  }
}

__device__ __forceinline__ int sel_cols(int ni_lim) {
  return ni_lim <= 0 ? SEL_SKIP : ni_lim == 1 ? SEL_NI1 : ni_lim == 2 ? SEL_NI2 : ni_lim == 3 ? SEL_NI3 : SEL_FULL;
}
__device__ __forceinline__ int sel_rows(int mi_lim) {  // mi_lim is even (n is padded to 16-row chunks)
  return mi_lim <= 0 ? SEL_SKIP : mi_lim == 2 ? SEL_MI2 : SEL_FULL;
}

// Geometry of this CTA's half tile inside the 128x128 tile.
struct HalfGeom {
  int r0h, c0h;   // tile-relative row / column offset of the half (0 or 64)
  int ncols;      // valid columns of the half (FWD_ROW tiles may be narrower than 64)
  int gcol_off;   // FWD_ROW: offset of the tile's first column inside the right-hand-side row (tc.j * colw)
};

// Consumer side of one half tile (warps 0-3).  RAGGED = the tile touches the padded tail of the last block row:
// only then are the DMMAs / loads / stores predicated per 8-row slab (mi < mi_valid); full tiles run the clean loop.
// BWD = the BWD_ROW tiles of k_tile_bwd (COLSPLIT, laid out like FWD_ROW); false compiles exactly the code of k_tile_gemm.
template <bool COLSPLIT, bool RAGGED, bool BWD = false>
__device__ __forceinline__ void consume_tile(const GemmArgs& g, const TileCoord& tc, const HalfGeom& hg, double* stages,
                                             double* rbuf, uint64_t* full, uint64_t* empty, uint64_t* rfull, uint64_t* rempty,
                                             int gp, int nchunks, int rows_valid) {
  constexpr int LDA = COLSPLIT ? LDS_T : LDS_H;   // A operand chunk: 128 rows (COLSPLIT) or 64
  constexpr int LDB = COLSPLIT ? LDS_H : LDS_T;   // B operand chunk: 64 rows (COLSPLIT) or 128
  constexpr int LDT = LDS_H;                      // parked half tile: k-major rows of 64
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t npad = g.npad;
  // Eight consumer warps with 32 x 32 register tiles, two per SMSP (warps w and w + 4 share SMSP w mod 4): a CTA that is
  // alone on its SM - the thin launches of small batches - still has a second warp per scheduler to fill the bubbles of
  // the first (barrier waits, fragment-load latency at chunk boundaries).
  // ROWSPLIT (64 x 128): 2 row groups x 4 column groups.  COLSPLIT (128 x 64): 4 row groups x 2 column groups.
  const int wm = COLSPLIT ? (warp >> 1) : (warp >> 2);
  const int wn = COLSPLIT ? (warp & 1) : (warp & 3);
  const int r0t = hg.r0h + wm * WROWS;       // tile-relative row of the warp tile's first row
  const int gq = lane >> 2, t = lane & 3;
  const bool fwd = BWD || g.mode == GEMM_FWD_ROW;
  // Column layout.  Default: column group wn owns the four 8-column blocks at 32 wn.  FWD_ROW tiles with fewer than 64
  // valid test columns (the reference predicts m = 100 test states per step: 64 + 36; narrow 32-column tiles when a
  // launch would otherwise have too few CTAs) use a compact layout: the nblk = ceil(ncols / 8) valid 8-column blocks are
  // dealt over the two column groups and every warp runs the chunk body specialised to its own block count - the
  // padding columns are neither multiplied nor loaded nor stored.
  int cbase = wn * 32, ni_lim = 4;
  if (COLSPLIT && fwd && hg.ncols < HB) {
    const int nblk = (hg.ncols + 7) >> 3, w0 = (nblk + 1) >> 1, w1 = nblk >> 1;
    ni_lim = wn == 0 ? w0 : w1;
    cbase = wn == 0 ? 0 : 8 * w0;
  }
  const int c0t = hg.c0h + cbase;             // tile-relative column of the warp tile's first column
  const int mi_valid = RAGGED ? min(MI_N, max(0, (rows_valid - r0t + 7) / 8)) : MI_N;
  const int row0 = wm * WROWS + gq;  // + mi*8 : A-operand row inside the chunk
  const int col0 = cbase + gq;    // + ni*8 : B-operand row inside the chunk

  // ---- operand traffic: ONE tensor-map TMA request (cp.async.bulk.tensor.3d, SASS UTMALDG) lands a whole operand chunk.
  // The box is KT columns x the PADDED row count (132 / 68), so the dense box pitch IS the bank-conflict-free padded
  // pitch of the fragment loads (the 4 extra rows per column are never read).  Round 1 issued one 1 KB bulk copy per
  // operand column (32 requests per chunk) from a dedicated producer warp; with two requests per chunk the issue is
  // folded into consumer warp 0: after it has released a stage it waits until the other seven warps have too and
  // refills it, its SMSP partner (warp 4) keeps the DMMA pipe busy meanwhile - no producer warpgroup, 128 registers
  // for every thread at two CTAs per SM.
  const CUtensorMap* mapA_L = COLSPLIT ? &g.tm_L132 : &g.tm_L68;
  const CUtensorMap* mapA_D = COLSPLIT ? &g.tm_DT132 : &g.tm_DT68;
  const CUtensorMap* mapB_L = COLSPLIT ? &g.tm_L68 : &g.tm_L132;
  const CUtensorMap* mapB_D = COLSPLIT ? &g.tm_DT68 : &g.tm_DT132;
  auto issue_main = [&](int c) {  // main-loop chunk c -> stage c % NSTAGE (called by lane 0 of warp 0)
    const int stage = c % NSTAGE, kb = tc.kb0 + c / (NB / KT), kc = kb * NB + (c % (NB / KT)) * KT;
    const CUtensorMap* ma; const CUtensorMap* mb; int ra, rb, gb = gp;
    if (kb == tc.a_diag_kb) { ma = mapA_D; ra = hg.r0h; }
    else { ma = mapA_L; ra = tc.i * NB + hg.r0h; }
    if (kb == tc.b_diag_kb) { mb = mapB_D; rb = hg.c0h; }
    else if (fwd) { mb = &g.tm_T68; rb = hg.gcol_off; gb = gp - g.t_gp_off; }
    else { mb = mapB_L; rb = tc.j * NB + hg.c0h; }
    double* dst = stages + stage * STAGE_DOUBLES;
    if (BWD) {  // A = L(k rows, i columns)^T: the box of KT rows x NB columns lands row-major, [column][KT]
      mbar_expect_tx(&full[stage], (KT * NB + KT * LDB) * sizeof(double));
      tma_load_3d(dst, &g.tm_LT, kc, tc.i * NB, gp, &full[stage]);
    } else {
      mbar_expect_tx(&full[stage], STAGE_DOUBLES * sizeof(double));
      tma_load_3d(dst, ma, ra, kc, gp, &full[stage]);
    }
    tma_load_3d(dst + KT * LDA, mb, rb, kc, gb, &full[stage]);
  };
  auto issue_r = [&](int c) {  // chunk c of the post-multiplier inv(L_rblk) -> rbuf[c % NRBUF]
    const int buf = c % NRBUF;
    mbar_expect_tx(&rfull[buf], RBUF_DOUBLES * sizeof(double));
    tma_load_3d(rbuf + buf * RBUF_DOUBLES, BWD ? &g.tm_DT132 : &g.tm_D132, 0, tc.rblk * NB + c * KT, gp, &rfull[buf]);
  };
  if (warp == 0 && lane == 0) {  // prologue: fill the ring, start the post-multiplier
    for (int c = 0; c < min(NSTAGE, nchunks); ++c) issue_main(c);
    if (tc.post) for (int c = 0; c < NRBUF; ++c) issue_r(c);
  }

  // The accumulators start at -Cin (Cholesky tiles: K(i,j); FWD_ROW: the right-hand-side block), loaded straight
  // into the accumulator registers while the first operand chunks are still in flight.  After the k-loop
  // acc = sum - Cin = -(Cin - sum); the sign is folded into the stores below.
  const int64_t grow = (int64_t)tc.i * NB, gcol = fwd ? (int64_t)hg.gcol_off : (int64_t)tc.j * NB;
  double acc[MI_N][4][2];
  if (fwd) {
    const double* Tin = g.Tm + (int64_t)(gp - g.t_gp_off) * g.t_stride + gcol + grow * g.ldt;
#pragma unroll
    for (int mi = 0; mi < MI_N; ++mi)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        const int r = r0t + mi * 8 + gq, cc = c0t + ni * 8 + 2 * t;
        double2 v = make_double2(0.0, 0.0);
        if ((!RAGGED || mi < mi_valid) && ni < ni_lim) v = *reinterpret_cast<const double2*>(Tin + cc + (int64_t)r * g.ldt);
        acc[mi][ni][0] = -v.x;
        acc[mi][ni][1] = -v.y;
      }
  } else if (tc.use_cin) {
    const double* Cin = g.Cin + (int64_t)gp * g.mat_stride + grow + gcol * npad;
#pragma unroll
    for (int mi = 0; mi < MI_N; ++mi)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        const int r = r0t + mi * 8 + gq, cc = c0t + ni * 8 + 2 * t;
        const bool ok = !RAGGED || mi < mi_valid;
        acc[mi][ni][0] = ok ? -Cin[r + (int64_t)cc * npad] : 0.0;
        acc[mi][ni][1] = ok ? -Cin[r + (int64_t)(cc + 1) * npad] : 0.0;
      }
  } else {
#pragma unroll
    for (int mi = 0; mi < MI_N; ++mi)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
  }

  // Triangular operands: the leading k-block of TRTRI_ROW (B = inv(L_jj)) and of LAUUM (A = inv(L_ii)^T) is
  // triangular, and CHOL_DIAG only needs the lower half of its symmetric tile.  The 8x8 DMMA blocks that would
  // multiply structural zeros (or compute the unused upper half) are skipped through compile-time specialised
  // chunk bodies (no per-DMMA predicates).  Ragged tiles (last block row) select the row-limited body.
#ifdef GPRB_TIMELINE
  long long tl_wait = 0;  // cycles this warp spent waiting for operand chunks in the main loop
#endif
  int npred = 0;
  if (g.mode == GEMM_LAUUM) npred = min(nchunks, NB / KT);
  else if (!RAGGED && (g.mode == GEMM_CHOL_DIAG || (g.mode == GEMM_CHOL_TRAIL && tc.i == tc.j))) npred = nchunks;
  else if (!RAGGED && g.mode == GEMM_TRTRI_ROW) npred = NB / KT;
  const int diag_off = (c0t - r0t) / 8;  // block (mi, ni) touches the lower triangle of the tile iff mi >= ni + diag_off
  // LAUUM diagonal tiles are symmetric: beyond the leading (triangular-operand) k-block only the 8x8 blocks on or below the
  // diagonal are accumulated, the store mirrors them into the upper half (the gradient stage reads whole tiles)
  // (decided per TILE: the mirror partner of a block may live in the other half, so a ragged tile - last block row - is
  // computed and stored in full by both of its halves, also by the half whose own rows are all valid)
  const bool lsym = rows_valid == NB && g.mode == GEMM_LAUUM && tc.i == tc.j;
  const int sel_tri = diag_off >= MI_N ? SEL_SKIP : diag_off == 0 ? SEL_TRI0 : SEL_FULL;  // diag_off is a multiple of 4
  const int sel_plain = ni_lim < 4 ? sel_cols(ni_lim) : sel_rows(mi_valid);  // column-limited bodies run all 8 row slabs
  {
    int stage = 0; uint32_t phase = 0;
    for (int c = 0; c < nchunks; ++c) {
#ifdef GPRB_TIMELINE
      const long long w0 = clock64();
      mbar_wait(&full[stage], phase);
      if (c > 0) tl_wait += clock64() - w0;  // the wait for the first chunk is the `fill` phase
#else
      mbar_wait(&full[stage], phase);
#endif
      if (c == 0) GPRB_TL(1);
      const double* As = stages + stage * STAGE_DOUBLES;
      int sel = sel_plain;
      if (c < npred) {
        if (g.mode == GEMM_LAUUM) sel = sel_rows(min(mi_valid, 2 * c + 2 - r0t / 8));  // rows r <= 16c + 15 of the triangular A
        else if (g.mode == GEMM_TRTRI_ROW) {                                           // columns <= 16c + 15 of the triangular B
          const int nl = 2 * c + 2 - c0t / 8;
          sel = nl <= 0 ? SEL_SKIP : nl == 2 ? SEL_NI2 : SEL_FULL;
        } else sel = sel_tri;
      } else if (lsym) sel = sel_tri;
      if (BWD) chunk_dispatch<LDA, LDB, 1, KT>(sel, acc, As + row0 * KT + t, As + KT * LDA + t * LDB + col0);
      else chunk_dispatch<LDA, LDB>(sel, acc, As + t * LDA + row0, As + KT * LDA + t * LDB + col0);
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[stage]);
      if (warp == 0 && c + NSTAGE < nchunks) {  // refill: every consumer warp has released this stage
        mbar_wait(&empty[stage], phase);
        if (lane == 0) issue_main(c + NSTAGE);
      }
      if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
    }
  }

  GPRB_TL(2);
#ifdef GPRB_TIMELINE
  if (g.tl && threadIdx.x == 0) g.tl[((int64_t)blockIdx.y * gridDim.x + blockIdx.x) * 8 + 7] = (unsigned long long)tl_wait;
#endif
  GPRB_TL(3);
  double* Cout = g.Cout + (int64_t)gp * g.mat_stride;
  if (tc.post == 0) {
    // CHOL_DIAG: S(j,j) -> Lm(j,j).  LAUUM: K^-1(i,j), i > j, goes un-transposed into the free upper tile (j,i) of A
    // (K stays intact in the lower tiles for the gradient stage); diagonal tiles go to the KinvD side buffer.
    double* out = Cout + grow + gcol * npad;
    int64_t ldo = npad;
    const double sgn = tc.use_cin ? -1.0 : 1.0;  // CHOL_DIAG: S = Cin - sum = -acc
    if (g.mode == GEMM_LAUUM) {
      if (tc.i != tc.j) out = Cout + gcol + grow * npad;
      else { out = g.KinvD + (int64_t)gp * g.dinv_stride + (int64_t)tc.i * NB * NB; ldo = NB; }
    }
#pragma unroll
    for (int mi = 0; mi < MI_N; ++mi)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        if (RAGGED && mi >= mi_valid) continue;
        if (lsym && mi < ni + diag_off) continue;  // upper 8x8 blocks hold partial sums only: written by their mirror block
        const int r = r0t + mi * 8 + gq, cc = c0t + ni * 8 + 2 * t;
        out[r + (int64_t)cc * ldo] = sgn * acc[mi][ni][0];
        out[r + (int64_t)(cc + 1) * ldo] = sgn * acc[mi][ni][1];
        if (lsym && mi > ni + diag_off)  // strictly-lower block: mirror (rows cc, cc + 1 of column r are adjacent)
          *reinterpret_cast<double2*>(&out[cc + (int64_t)r * ldo]) = make_double2(acc[mi][ni][0], acc[mi][ni][1]);
      }
    GPRB_TL(6);
    return;
  }

  // ---- post-multiply: park T in the (now idle) stage ring, then a second DMMA pass against Dinv chunks
  named_bar_sync(1, N_CONSUMER_WARPS * 32);  // every consumer finished reading the ring
  double* Ts = stages;
  if (tc.post == 1) {  // ROWSPLIT.  A operand: Ts[k][m] = T[m][k], m = the half's 64 rows, k = the tile's 128 columns
#pragma unroll
    for (int mi = 0; mi < MI_N; ++mi)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        const int r = wm * WROWS + mi * 8 + gq, cc = cbase + ni * 8 + 2 * t;
        const bool ok = !RAGGED || mi < mi_valid;  // skipped rows are parked as zeros (finite operands for the second pass)
        Ts[cc * LDT + r] = ok ? acc[mi][ni][0] : 0.0;
        Ts[(cc + 1) * LDT + r] = ok ? acc[mi][ni][1] : 0.0;
      }
  } else {  // COLSPLIT.  B operand: Ts[k][n] = T[k][n], k = the tile's 128 rows, n = the half's 64 columns
#pragma unroll
    for (int mi = 0; mi < MI_N; ++mi)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        const int r = wm * WROWS + mi * 8 + gq, cc = cbase + ni * 8 + 2 * t;
        const bool ok = !RAGGED || mi < mi_valid;
        if (ni < ni_lim) *reinterpret_cast<double2*>(&Ts[r * LDT + cc]) = ok ? make_double2(acc[mi][ni][0], acc[mi][ni][1]) : make_double2(0.0, 0.0);
      }
  }
#pragma unroll
  for (int mi = 0; mi < MI_N; ++mi)
#pragma unroll
    for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
  named_bar_sync(1, N_CONSUMER_WARPS * 32);
  GPRB_TL(4);

  // Dinv is lower triangular: R[x][k] == 0 for k > x.  post 1: x = output column, post 2: x = output row
  // (tile-relative; the post-multiplier chunk c covers k = 16c .. 16c + 15 of the whole tile).
  // BWD: R = DinvT is upper triangular, R[x][k] == 0 for k < x: chunk c only meets the rows x <= 16c + 15.
  const int kmax = (tc.post == 1) ? (c0t + 31) : BWD ? rows_valid - 1 : min(r0t + WROWS - 1, rows_valid - 1);
  for (int c = 0; c < NB / KT; ++c) {
    const int buf = c % NRBUF;
    mbar_wait(&rfull[buf], (c / NRBUF) & 1);
    if (BWD) {
      if (c * KT <= kmax && c * KT + KT - 1 >= r0t) {
        const double* Rs = rbuf + buf * RBUF_DOUBLES + t * LDS_T;
        const double* Tc = Ts + (c * KT + t) * LDT;
        const int sel = (sel_plain == SEL_FULL && 2 * c == r0t / 8) ? SEL_MI2 : sel_plain;  // rows r0t + 16 .. lie below chunk c
        chunk_dispatch<LDA, LDB>(sel, acc, Rs + r0t + gq, Tc + col0);
      }
    } else if (c * KT <= kmax) {
      const double* Rs = rbuf + buf * RBUF_DOUBLES + t * LDS_T;
      const double* Tc = Ts + (c * KT + t) * LDT;
      // triangular skip inside the warp tile: chunk c only meets output columns (post 1) / rows (post 2) x >= 16 c
      int sel = sel_plain;
      if (tc.post == 1) {  // out(64 x 128) = T(64 x 128) * R^T : A = parked T (64-wide rows), B = R chunk (128-wide rows)
        if (sel_plain == SEL_FULL && 2 * c - c0t / 8 == 2) sel = SEL_NLO2;
        chunk_dispatch<LDA, LDB>(sel, acc, Tc + row0, Rs + c0t + gq);
      } else {             // out(128 x 64) = R(128 x 128) * T(128 x 64) : A = R chunk (128-wide rows), B = parked T (64-wide rows)
        const int lo = 2 * c - r0t / 8;  // first 8-row slab that meets chunk c: 0 or 2 here (c * KT <= kmax)
        if (lo > 0) {
          if (sel_plain == SEL_FULL) sel = SEL_MLO2;
          else if (sel_plain == SEL_NI3) sel = SEL_MLO2_NI3;
        }
        chunk_dispatch<LDA, LDB>(sel, acc, Rs + r0t + gq, Tc + col0);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&rempty[buf]);
    if (warp == 0 && c + NRBUF < NB / KT) {
      mbar_wait(&rempty[buf], (c / NRBUF) & 1);
      if (lane == 0) issue_r(c + NRBUF);
    }
  }
  GPRB_TL(5);

  if (tc.post == 1) {
#pragma unroll
    for (int mi = 0; mi < MI_N; ++mi)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        if (RAGGED && mi >= mi_valid) continue;
        const int r = r0t + mi * 8 + gq, cc = c0t + ni * 8 + 2 * t;
        Cout[grow + r + (gcol + cc) * npad] = -acc[mi][ni][0];      // parked operand was -(Cin - sum)
        Cout[grow + r + (gcol + cc + 1) * npad] = -acc[mi][ni][1];
      }
  } else {  // W(i,j) = -acc, stored transposed as V(j,i); FWD_ROW (parked operand sum - T(i,:)): row r of the solved block
    double* outp = fwd ? g.Tm + (int64_t)(gp - g.t_gp_off) * g.t_stride + gcol + grow * g.ldt : Cout + gcol + grow * npad;
    const int64_t ldo = fwd ? g.ldt : npad;
#pragma unroll
    for (int mi = 0; mi < MI_N; ++mi)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        if ((RAGGED && mi >= mi_valid) || ni >= ni_lim) continue;
        const int r = r0t + mi * 8 + gq, cc = c0t + ni * 8 + 2 * t;
        *reinterpret_cast<double2*>(&outp[cc + r * ldo]) = make_double2(-acc[mi][ni][0], -acc[mi][ni][1]);
      }
  }
  GPRB_TL(6);
}

// COLSPLIT = false: 64 x 128 halves (CHOL_*, LAUUM); true: 128 x 64 halves (TRTRI_ROW) / <= 64-column tiles (FWD_ROW,
// BWD_ROW).
template <bool COLSPLIT, bool BWD>
__device__ __forceinline__ void tile_gemm_body(const GemmArgs& g) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* stages = reinterpret_cast<double*>(smem_raw);
  double* rbuf = stages + NSTAGE * STAGE_DOUBLES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(rbuf + NRBUF * RBUF_DOUBLES);
  uint64_t* full = bars;            // [NSTAGE]
  uint64_t* empty = bars + NSTAGE;  // [NSTAGE]
  uint64_t* rfull = bars + 2 * NSTAGE;            // [NRBUF]
  uint64_t* rempty = bars + 2 * NSTAGE + NRBUF;   // [NRBUF]

  GPRB_TL(0);
  const int gp = g.list ? g.list[blockIdx.y] : g.gp_off + blockIdx.y;
  // A GP whose factorisation already hit a non-positive pivot (make_posdef! will retry it with more jitter) skips the
  // rest of the failed attempt, like dpotrf stopping at the failing column.  The load overlaps the setup below.
  const int failed = g.fail ? g.fail[gp] : 0;
  const bool fwd = BWD || g.mode == GEMM_FWD_ROW;
  // blockIdx.x: (tile, half) for every mode but FWD_ROW / BWD_ROW, whose tiles are already <= 64 columns wide
  const int half = fwd ? 0 : (int)(blockIdx.x & 1);
  TileCoord tc;
  if (BWD) {
    tc.i = g.step; tc.j = blockIdx.x; tc.kb0 = g.step + 1; tc.kb1 = g.J; tc.a_diag_kb = tc.b_diag_kb = -1;
    tc.use_cin = true; tc.post = 2; tc.rblk = g.step;
  } else {
    tc = tile_coord(g.mode, g.step, g.J, g.row0, fwd ? (int)blockIdx.x : (int)(blockIdx.x >> 1));
  }
  HalfGeom hg;
  hg.r0h = COLSPLIT ? 0 : half * HB;
  hg.c0h = COLSPLIT ? (fwd ? 0 : half * HB) : 0;
  hg.ncols = fwd ? min(g.colw, g.ncols - tc.j * g.colw) : HB;
  hg.gcol_off = fwd ? tc.j * g.colw : 0;

  // Padding skip: rows/cols >= nv (n rounded up to the 16-wide chunk) are never computed and never read.
  // Only the last block row / the last k-block are ragged.
  const int nvl = g.nv - (g.J - 1) * NB;                          // valid rows of the last 128-block (multiple of 16)
  const int last_kb_chunks = nvl / KT;                             // chunks of k-block J-1 that hold valid k
  const int nchunks = (tc.kb1 - tc.kb0) * (NB / KT) - ((tc.kb1 == g.J && tc.kb1 > tc.kb0) ? (NB / KT - last_kb_chunks) : 0);
  const int rows_valid = (tc.i == g.J - 1) ? nvl : NB;            // valid output rows of this tile
  // a row half that lies entirely in the padding of the last block row has nothing to compute (uniform over the CTA)
  if (failed != 0 || (!COLSPLIT && hg.r0h >= rows_valid)) return;
  // The K half tile the accumulators start from is read by per-thread loads in the DMMA accumulator layout: 64-byte pieces,
  // one DRAM page each.  Eight TMA prefetch requests (64 rows x 16 columns: 512-byte pieces) pull it into L2 first; the
  // register loads below then merge with / hit those lines.
  if (!COLSPLIT && g.pf_cin && tc.use_cin && threadIdx.x == 32) {
#pragma unroll
    for (int q = 0; q < NB / KT; ++q) tma_prefetch_3d(&g.tm_A68, tc.i * NB + hg.r0h, tc.j * NB + q * KT, gp);
  }

  if (threadIdx.x == 0) {
    for (int s = 0; s < NSTAGE; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], N_CONSUMER_WARPS); }
    for (int s = 0; s < NRBUF; ++s) { mbar_init(&rfull[s], 1); mbar_init(&rempty[s], N_CONSUMER_WARPS); }
    mbar_fence_init();
  }
  __syncthreads();

  // RAGGED whenever the warp tiles of this half do not all have 64 valid rows
  const int rows_here = rows_valid - hg.r0h;  // valid rows from the half's first row on (ROWSPLIT: up to 64 matter)
  const bool ragged = COLSPLIT ? (rows_valid < NB) : (rows_here < HB);
  if (!ragged) consume_tile<COLSPLIT, false, BWD>(g, tc, hg, stages, rbuf, full, empty, rfull, rempty, gp, nchunks, rows_valid);
  else consume_tile<COLSPLIT, true, BWD>(g, tc, hg, stages, rbuf, full, empty, rfull, rempty, gp, nchunks, rows_valid);
}

template <bool COLSPLIT>
__global__ void __launch_bounds__(GEMM_THREADS, 2) k_tile_gemm(const __grid_constant__ GemmArgs g) {
  tile_gemm_body<COLSPLIT, false>(g);
}

// GEMM_BWD_ROW tiles (the backward block substitution of the predictive gradient), a kernel of their own so that the
// modes of k_tile_gemm keep their code.
__global__ void __launch_bounds__(GEMM_THREADS, 2) k_tile_bwd(const __grid_constant__ GemmArgs g) {
  tile_gemm_body<true, true>(g);
}

// The dynamic shared-memory opt-in is a per-device function attribute: gprb_init calls this for the device of every
// context it creates (a process-wide "configured" flag would leave a second GPU of the same process un-opted-in).
int configure_tile_gemm() {
  cudaError_t e = cudaFuncSetAttribute(k_tile_gemm<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GEMM_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tile_gemm<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GEMM_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tile_gemm<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tile_gemm<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tile_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GEMM_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tile_bwd, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_tile_gemm)", __FILE__, __LINE__);
  return 0;
}

// ntiles = logical tiles of the launch: 128x128 tiles for every mode but FWD_ROW / BWD_ROW (each becomes two CTAs), column
// tiles of g.colw <= 64 test columns for FWD_ROW / BWD_ROW (one CTA each).
int launch_tile_gemm(const GemmArgs& g, int ntiles, int count, cudaStream_t stream) {
  if (ntiles <= 0 || count <= 0) return 0;
  const bool colsplit = g.mode == GEMM_TRTRI_ROW || g.mode == GEMM_FWD_ROW;
  const bool rhs = g.mode == GEMM_FWD_ROW || g.mode == GEMM_BWD_ROW;
  if (rhs && (g.colw > HB || g.colw < 8 || (g.colw & 7))) {
    set_error("k_tile_gemm: FWD_ROW / BWD_ROW tiles are at most 64 columns wide");
    return GPRB_ERR_ARG;
  }
  dim3 grid(rhs ? ntiles : 2 * ntiles, count);
  if (g.mode == GEMM_BWD_ROW) k_tile_bwd<<<grid, GEMM_THREADS, GEMM_SMEM, stream>>>(g);
  else if (colsplit) k_tile_gemm<true><<<grid, GEMM_THREADS, GEMM_SMEM, stream>>>(g);
  else k_tile_gemm<false><<<grid, GEMM_THREADS, GEMM_SMEM, stream>>>(g);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_tile_gemm launch", __FILE__, __LINE__);
  return 0;
}

}  // namespace gprb
