// Damped normal-equation solve + manifold update kernels (sm_100a).
//
// Replaces what ceres::Solve does between two Jacobian evaluations for the reference's spline problem
// (SplineTrajectoryEstimator::Optimize, include/OpenCameraCalibrator/core/spline_trajectory_estimator.impl.h:254-276):
//   * Jacobi column scaling + Levenberg-Marquardt diagonal  (Ceres TrustRegionMinimizer / LevenbergMarquardtStrategy)
//   * SPARSE_NORMAL_CHOLESKY on (J^T J + D^T D)              -> exact LDL^T of the banded (spline knots, time ordered)
//     + bordered (T_i_c, gravity, line delay, bias knots) system: the spline control points are Schur-eliminated first
//   * LieLocalParameterization::Plus on every SO(3) knot and on T_i_c (basalt_spline/ceres_local_param.h:84-92)
//
// The band factorisation is a recurrence along time, so it is reordered by nested dissection of the time axis:
//   level 0   the knot columns are cut into P time chunks separated by P-1 separators of kd columns; every chunk's interior
//             is eliminated in parallel (one CTA per chunk, blocked LDL^T in a circular shared-memory window, FP64 tensor-core
//             trailing updates), carrying the couplings to its two separators, the border and the right-hand side;
//   level l   the separators form a block-tridiagonal system: block cyclic reduction eliminates every other block in
//             parallel (same elimination routine, one CTA per block), halving the block count per level;
//   root      one CTA factors the last block + the border (T_i_c, gravity, line delay, bias knots, ...) and solves them;
// then the back-substitution walks the levels in reverse.  The sequential pivot chain is O(nk / P + kd log P) columns instead
// of nk.  The last kernel forms the step and the model cost change.
#include "icc_device_math.cuh"
#include "icc_kernels.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace icc {

void count_launch();

namespace {

constexpr int NT = 512;          // threads of the factorisation kernels

// Programmatic dependent launch: every solver kernel is launched with programmatic stream serialisation, does the work that
// does not depend on its predecessor (shared-memory set-up, zero fill) first, then waits for the predecessor's results.  The
// "launch dependents" trigger is issued right AFTER the wait, so when a kernel starts, everything older than its direct
// predecessor is already complete and visible.
__device__ __forceinline__ void pdl_wait_then_trigger() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
template <class... KArgs, class... Args>
void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
constexpr int MAX_LEVELS = 12;

struct SolvePlan {
  int P, w;                       // level-0 chunks, separator width (0 when P == 1)
  int len, rem;                   // chunk c owns len + (c < rem) interior columns
  int L;                          // cyclic-reduction levels 1..L; reduced system R_l has S[l] blocks of w columns (l = 1..L+1)
  int S[MAX_LEVELS + 2], off[MAX_LEVELS + 2];   // off[l]: first column of R_l inside the concatenated reduced arrays
  int nkr_total;                  // columns of all reduced systems together
  int kdr, ldbr;                  // reduced systems: half bandwidth 2w-1, column length
  int nbl;                        // local border rows of an elimination: w + nb + 1 (left separator | border | rhs)
  int WS_A, WS_R, WS_B;           // window slots (power of two): level 0, cyclic-reduction levels, root
  int cl_global, cs_global;       // wide borders: the level-0 local border block / the root's border block live in HBM (L2), not in shared memory
  int stage0;                     // level-0 back-substitution stages its El rows in shared memory
  int valid;                      // 0: no plan fits the shared-memory limits
};
__host__ __device__ inline int chunk_a(const SolvePlan& pl, int c) { return c * (pl.len + pl.w) + (c < pl.rem ? c : pl.rem); }
__host__ __device__ inline int chunk_b(const SolvePlan& pl, int c) { return chunk_a(pl, c) + pl.len + (c < pl.rem ? 1 : 0); }
// block j of R_l is the original separator ((j+1) << (l-1)) - 1, which sits right behind the interior of that chunk
__host__ __device__ inline int sep_col(const SolvePlan& pl, int l, int j) { return chunk_b(pl, ((j + 1) << (l - 1)) - 1); }

// Workspace (doubles): Lb[nk*ldb] | El[nk*nbl] | y[n] | R{bandr[nkr_total*ldbr] | Er[nkr_total*nbp] | Cr[nbp*nbp]} | Lbr | Elr[nkr_total*nbl] | Wg
struct SolveWs { double *Lb, *El, *y, *bandr, *Er, *Cr, *Lbr, *Elr, *Wg, *Clg, *Csg; size_t reduced_doubles, total; };
__host__ __device__ inline SolveWs carve(double* ws, int nk, int nb, int ldb, const SolvePlan& pl) {
  SolveWs w; const int nbp = nb + 1; const size_t n = (size_t)nk + nb, nr = (size_t)pl.nkr_total;
  w.Lb = ws; w.El = w.Lb + (size_t)nk * ldb; w.y = w.El + (size_t)nk * pl.nbl;
  w.bandr = w.y + ((n + 3) & ~(size_t)3); w.Er = w.bandr + nr * pl.ldbr; w.Cr = w.Er + nr * nbp;
  w.reduced_doubles = nr * pl.ldbr + nr * nbp + (size_t)nbp * nbp;
  w.Lbr = w.Cr + (size_t)nbp * nbp; w.Elr = w.Lbr + nr * pl.ldbr;
  w.Wg = w.Elr + nr * pl.nbl;                                       // nk x (kd + KB + nbl): pre-scaled window columns of level 0
  w.Clg = w.Wg + (size_t)nk * (ldb - 1 + 8 + pl.nbl);               // P x nbl^2 (only when cl_global)
  w.Csg = w.Clg + (pl.cl_global ? (size_t)pl.P * pl.nbl * pl.nbl : 0);  // nbp^2 (only when cs_global)
  w.total = (size_t)(w.Csg + (pl.cs_global ? (size_t)nbp * nbp : 0) - ws) + 16;
  return w;
}

__device__ __forceinline__ int tri_row(int idx) {   // idx = r(r+1)/2 + c, 0 <= c <= r  ->  r
  int r = (int)((sqrtf(8.0f * (float)idx + 1.0f) - 1.0f) * 0.5f);   // estimate, made exact by the two loops
  while ((r + 1) * (r + 2) / 2 <= idx) ++r;
  while (r * (r + 1) / 2 > idx) --r;
  return r;
}

// LM diagonal: clamp(diag(S H S), min, max) / radius   (LevenbergMarquardtStrategy::ComputeStep)
__device__ __forceinline__ double lm_d2(const DeviceProblem& P, const double* scale, const SolveParams& sp, int i) {
  const double d = i < P.nk ? P.ne[(int64_t)i * P.ldb] : P.ne[P.ne_off_C + (int64_t)(i - P.nk) * P.nb + (i - P.nk)];
  const double s = scale[i];
  return fmin(fmax(d * s * s, sp.min_diag), sp.max_diag) / sp.radius;
}

constexpr int KB = 8;             // panel width of the blocked LDL^T

// Blocked right-looking LDL^T inside a circular shared-memory window.
//
// Window column layout (CL doubles): [band part, ldbp = kd + KB entries, offsets > kd are zero padding][local border rows, nbl].
// Per panel of KB columns:
//   (1) KB sequential column steps that only update the OTHER PANEL columns (<= (KB-1)(kd+1+nbl) entries, 1 sync each);
//   (2) ONE rank-KB update of the trailing window + dense local-border block, done as a symmetric GEMM on the FP64 tensor
//       cores: with M = kd + nbl trailing positions (the kd band columns after the panel, then the border rows),
//       T[x][y] -= sum_jj L[x][jj] L[y][jj] / D_jj,  L[x][jj] = entry of panel column jj at trailing position x,
//       tiled in 8x8 blocks of m8n8k4 DMMAs (KB/4 k-steps).  Thanks to the zero padding no operand needs a bounds test.
__device__ __forceinline__ void dmma_acc(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}
// lower-triangular list of 8x8 blocks (bi >= bj) covering M trailing positions
__device__ int build_block_table(uchar2* blocks, int M) {   // the nbk blocks of block-column 0 come first (look-ahead order)
  const int nbk = (M + 7) / 8, n = nbk * (nbk + 1) / 2;
  for (int idx = threadIdx.x; idx < n; idx += blockDim.x) {
    if (idx < nbk) { blocks[idx] = make_uchar2(idx, 0); continue; }
    const int k = idx - nbk, r = tri_row(k), c = k - r * (r + 1) / 2;     // lower triangle of the (nbk-1)^2 remainder
    blocks[idx] = make_uchar2(r + 1, c + 1);
  }
  return n;
}
struct FactorSmem { double* W; double* Cl; uchar2* blocks; int nblocks; double* Ld; double* inv; int* flag; int nbl; };   // Ld, inv: double-buffered by panel parity

// (a)+(b) of one panel, executed by ONE warp (no block-wide barrier inside):
//   (a) lane 0 factors the KB x KB diagonal block in registers (unit-lower l, pivots D -> inv), kb <= KB columns are pivots;
//   (b) every lane forward-substitutes the KB panel entries of its trailing rows x (x = lane, lane+32, ...) against l.
// Reciprocal of a positive pivot on the critical path of the factorisation: single-precision hardware seed (MUFU.RCP) +
// two FP64 Newton steps (4 dependent FMAs, <= 2 ulp) instead of the ~2x longer correctly-rounded division sequence.
// Pivots outside the float range fall back to the exact division.
__device__ __forceinline__ double fast_rcp(double d) {
  if (!(d > 1e-30 && d < 1e30)) return 1.0 / d;
  double r = (double)__frcp_rn((float)d);
  double e = fma(-d, r, 1.0); r = fma(r, e, r);
  e = fma(-d, r, 1.0); r = fma(r, e, r);
  return r;
}

constexpr int PW = 3;   // warps cooperating on a panel factorisation (96 lanes >= typical M = kd + nbl rows)
__device__ __forceinline__ void panel_factor_warp(const FactorSmem& fs, int jp, int kb, int kd, int ldbp, int CL, int mask, int buf) {
  const int lane = threadIdx.x & 31, M = kd + fs.nbl, gl = threadIdx.x;   // gl = lane index within the PW-warp group (warps 0..PW-1)
  double* W = fs.W;
  double* inv = fs.inv + buf * KB;
  double* Ld = fs.Ld + buf * KB * KB;
  double* pc[KB];
#pragma unroll
  for (int c = 0; c < KB; ++c) pc[c] = W + (size_t)((jp + c) & mask) * CL;
  if (gl == 0) {
    double a[KB][KB], ivr[KB];
#pragma unroll
    for (int c = 0; c < KB; ++c)
#pragma unroll
      for (int r = c; r < KB; ++r) a[r][c] = pc[c][r - c];
    bool ok = true;
#pragma unroll
    for (int j = 0; j < KB; ++j) {
      if (j < kb) {
        const double D = a[j][j];
        if (!(D > 0.0) || !isfinite(D)) ok = false;
        ivr[j] = 1.0 / D;
#pragma unroll
        for (int c = j + 1; c < KB; ++c) {
          const double lcj = a[c][j] * ivr[j];
#pragma unroll
          for (int i = c; i < KB; ++i) a[i][c] = fma(-a[i][j], lcj, a[i][c]);
        }
      } else ivr[j] = 0.0;                                       // short last panel: missing columns contribute nothing
    }
#pragma unroll
    for (int c = 0; c < KB; ++c) {
      inv[c] = ivr[c];
#pragma unroll
      for (int r = c; r < KB; ++r) { pc[c][r - c] = a[r][c]; if (r > c) Ld[r * KB + c] = a[r][c] * ivr[c]; }
    }
    if (!ok) *fs.flag = 0;
  }
  asm volatile("bar.sync 1, %0;" :: "r"(PW * 32) : "memory");   // named barrier among the PW panel warps only
  // (b) rows below the block: w_rc = a_rc - sum_{k < min(c, kb)} w_rk l_ck   (l_ck = 0 for k >= kb)
  double lreg[KB * (KB - 1) / 2];
  {
    int q = 0;
#pragma unroll
    for (int c = 1; c < KB; ++c)
#pragma unroll
      for (int k = 0; k < c; ++k) lreg[q++] = Ld[c * KB + k];
  }
  for (int x = gl; x < M; x += PW * 32) {
    const bool band = x < kd;
    const int off = band ? KB + x : ldbp + x - kd;             // band rows: offset from column c is off - c
    double wv[KB];
#pragma unroll
    for (int c = 0; c < KB; ++c) wv[c] = pc[c][band ? off - c : off];
    int q = 0;
#pragma unroll
    for (int c = 1; c < KB; ++c) {
      double v = wv[c];
#pragma unroll
      for (int k = 0; k < c; ++k) v = fma(-wv[k], lreg[q++], v);
      wv[c] = v;
      if (!band || off - c <= kd) pc[c][band ? off - c : off] = v;   // never touch the zero padding
    }
  }
}

// rank-KB tensor-core update of trailing blocks [b_begin, b_end) of the block table with the finished panel at jp
__device__ __forceinline__ void trailing_blocks(const FactorSmem& fs, int jp, int kd, int ldbp, int CL, int mask, int buf, int b_begin, int b_end, int wslot, int nslots) {
  const int lane = threadIdx.x & 31, fr = lane >> 2, fk = lane & 3, M = kd + fs.nbl;
  double* W = fs.W;
  const double* inv = fs.inv + buf * KB;
  for (int bidx = b_begin + wslot; bidx < b_end; bidx += nslots) {
    const int bi = fs.blocks[bidx].x, bj = fs.blocks[bidx].y;   // bi >= bj
    const int xa = 8 * bi + fr, xb = 8 * bj + fr;
    double acc[2] = {0.0, 0.0};
#pragma unroll
    for (int ks = 0; ks < KB / 4; ++ks) {
      const int jj = 4 * ks + fk;
      const double* cj = W + (size_t)((jp + jj) & mask) * CL;
      const double la = xa < kd ? cj[KB + xa - jj] : (xa < M ? cj[ldbp + xa - kd] : 0.0);
      const double lb = xb < kd ? cj[KB + xb - jj] : (xb < M ? cj[ldbp + xb - kd] : 0.0);
      dmma_acc(acc, -la * inv[jj], lb);
    }
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int y = 8 * bj + 2 * fk + e;
      if (xa >= y && xa < M) {
        double* dst = y < kd ? W + (size_t)((jp + KB + y) & mask) * CL + (xa < kd ? xa - y : ldbp + xa - kd) : fs.Cl + (xa - kd) * fs.nbl + (y - kd);
        *dst += acc[e];
      }
    }
  }
}

// LDL^T elimination of columns [j_begin, j_end).  load(col, e) returns the (scaled, damped) original entry e of column col
// (0 outside the matrix AND for the padding offsets kd < e < ldbp); store(col, e, v) receives every finished column
// (unscaled storage: entry 0 = pivot D_j, others = L_ij D_j).  On return the window holds the updated columns >= j_end.
// Schedule per panel p (two block-wide barriers, look-ahead of depth one):
//   1. all warps: tensor-core update of the trailing blocks in block-column 0 (= the columns of panel p+1)     | barrier
//   2. warps 0..PW-1: factor panel p+1 (panel_factor_warp)  ||  other warps: remaining trailing blocks of panel p | barrier
// so the sequential pivot chain of panel p+1 overlaps the bulk of panel p's rank-KB update.
// The block table is ordered with the block-column-0 blocks first (build_block_table).
template <class Load, class Store>
__device__ bool factor_range(const FactorSmem& fs, int j_begin, int j_end, int kd, int ldbp, int CL, int WS, Load load, Store store) {
  const int tid = threadIdx.x, nt = blockDim.x, mask = WS - 1, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
  const int PB = ((WS - kd - KB) / KB) * KB, M = kd + fs.nbl, ncol0 = (M + 7) / 8;   // ncol0 = blocks with bj == 0
  double* W = fs.W;
  if (tid == 0) *fs.flag = 1;
  for (int j0 = j_begin; j0 < j_end; j0 += PB) {
    const int gend = min(j0 + PB, j_end);
    const int first = j0 == j_begin ? j_begin : j0 + kd + KB, last = gend + kd + KB;   // columns the group reads or updates
    {   // group load with 8 independent global loads in flight per thread; (column, entry) advance incrementally (no divisions)
      const int total = (last - first) * CL, de = nt % CL, dc = nt / CL;
      int e = tid % CL, col = first + tid / CL;
      for (int b0 = tid; b0 < total; b0 += 8 * nt) {
        double v[8]; int slot[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const bool in = b0 + u * nt < total;
          v[u] = in ? load(col, e) : 0.0;
          slot[u] = in ? (col & mask) * CL + e : -1;
          e += de; col += dc; if (e >= CL) { e -= CL; ++col; }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) if (slot[u] >= 0) W[slot[u]] = v[u];
      }
    }
    __syncthreads();
    if (warp < PW) panel_factor_warp(fs, j0, min(KB, gend - j0), kd, ldbp, CL, mask, 0);   // prologue: first panel of the group
    __syncthreads();
    if (*fs.flag == 0) return false;                            // uniform
    int buf = 0;
    for (int jp = j0; jp < gend; jp += KB, buf ^= 1) {
      const bool has_next = jp + KB < gend;
      trailing_blocks(fs, jp, kd, ldbp, CL, mask, buf, 0, ncol0, warp, nwarps);
      __syncthreads();
      if (warp < PW) { if (has_next) panel_factor_warp(fs, jp + KB, min(KB, gend - jp - KB), kd, ldbp, CL, mask, buf ^ 1); }
      if (warp >= PW || !has_next) trailing_blocks(fs, jp, kd, ldbp, CL, mask, buf, ncol0, fs.nblocks, has_next ? warp - PW : warp, has_next ? nwarps - PW : nwarps);
      __syncthreads();
      if (*fs.flag == 0) return false;                          // uniform
    }
    for (int col = j0 + warp; col < gend; col += nwarps) { const double* src = W + (size_t)(col & mask) * CL; for (int e = lane; e < CL; e += 32) store(col, e, src[e]); }
    __syncthreads();
  }
  return true;
}

// Descending back-substitution of the band part, driven by ONE warp whose registers hold the sliding window of pending
// right-hand sides (32*NR >= kd + 1 slots); x_j is broadcast with a shuffle, so the per-column dependency chain is
// select -> SHFL -> DMUL -> DFMA instead of shared-memory round trips.  tw[col - base] holds t on entry and x on exit.
// Columns >= unknown_end are known values (x = t, no pivot) that only scatter into the unknown ones.
template <int NR>
__device__ void backsub_warp(const double* __restrict__ Lb_g, double* tw, double* Bw, int base, int top, int unknown_end, int kd, int ldb, int PB, bool prestaged) {
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, win = 32 * NR;
  double t[NR]; int r[NR];
  if (tid < 32) {
#pragma unroll
    for (int k = 0; k < NR; ++k) {
      int rr = ((top - 1 - lane - 32 * k) % win + win) % win;   // distance from column top-1 to this slot's column
      r[k] = rr; const int col = top - 1 - rr;
      t[k] = col >= base ? tw[col - base] : 0.0;
    }
  }
  double* ipv = Bw + (size_t)(PB + kd) * ldb;                    // reciprocal pivots of the group (filled by all threads)
  for (int hi = top; hi > base; hi -= PB) {
    const int lo_own = max(base, hi - PB), lo = max(base, lo_own - kd);
    if (!prestaged) {   // contiguous copy of the factor columns [lo, hi) with 8 loads in flight per thread
      const int total = (hi - lo) * ldb, lim = (min(hi, unknown_end) - lo) * ldb;
      const double* src = Lb_g + (int64_t)lo * ldb;
      for (int b0 = tid; b0 < total; b0 += 8 * nt) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int idx = b0 + u * nt; v[u] = idx < lim ? src[idx] : 0.0; }
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int idx = b0 + u * nt; if (idx < total) Bw[idx] = v[u]; }
      }
      for (int idx = tid; idx < hi - lo_own; idx += nt) { const int col = lo_own + idx; ipv[idx] = col < unknown_end ? 1.0 / Lb_g[(int64_t)col * ldb] : 1.0; }
    }
    __syncthreads();
    if (tid < 32) {
      // L_{j, c} D_c of slot column c = j - r sits at Bw[(c - lo) * ldb + r]; as j decreases with c fixed, r decreases too,
      // so the address just walks down by one double per step
      const double* p[NR];
#pragma unroll
      for (int k = 0; k < NR; ++k) p[k] = Bw + (int64_t)(hi - 1 - r[k] - lo) * ldb + r[k];
      // value that enters this lane's slot when the lane next owns a column (column c enters after column c + win resolved):
      // fetched with one non-divergent vector load per 32 columns instead of a divergent load on the critical path
      double tnext = 0.0;
      { const int c_own = ((hi - 1) & ~31) + lane - win; tnext = (c_own >= base && c_own + win <= hi - 1) ? tw[c_own - base] : 0.0; }
      for (int j = hi - 1; j >= lo_own; --j) {
        double l[NR];
#pragma unroll
        for (int k = 0; k < NR; ++k) l[k] = ((unsigned)(r[k] - 1) < (unsigned)kd && j - r[k] >= base) ? *p[k] : 0.0;
        const double ipiv = ipv[j - lo_own];
        const int reg = (j & (win - 1)) >> 5;
        const bool owner = lane == (j & 31);
        double v = t[0];
#pragma unroll
        for (int k = 1; k < NR; ++k) if (k == reg) v = t[k];
        const double xj = __shfl_sync(0xffffffffu, v, j & 31) * ipiv;
#pragma unroll
        for (int k = 0; k < NR; ++k) t[k] = (owner && k == reg) ? tnext : fma(-l[k], xj, t[k]);
        if (owner) tw[j - base] = xj;
#pragma unroll
        for (int k = 0; k < NR; ++k) {
          if (r[k] == 0) { r[k] = win - 1; p[k] = Bw + (int64_t)(j - win - lo) * ldb + (win - 1); }   // slot re-assigned to column j - win (only read once r <= kd)
          else { --r[k]; --p[k]; }
        }
        if ((j & 31) == 0 && j > lo_own) { const int c_own = j - 32 + lane - win; tnext = c_own >= base ? tw[c_own - base] : 0.0; }   // next 32-column block
      }
    }
    __syncthreads();
  }
}
__device__ void backsub_dispatch(const double* Lb_g, double* tw, double* Bw, int base, int top, int unknown_end, int kd, int ldb, int PB, bool prestaged = false) {
  if (kd < 32) backsub_warp<1>(Lb_g, tw, Bw, base, top, unknown_end, kd, ldb, PB, prestaged);
  else if (kd < 64) backsub_warp<2>(Lb_g, tw, Bw, base, top, unknown_end, kd, ldb, PB, prestaged);
  else if (kd < 128) backsub_warp<4>(Lb_g, tw, Bw, base, top, unknown_end, kd, ldb, PB, prestaged);
  else backsub_warp<8>(Lb_g, tw, Bw, base, top, unknown_end, kd, ldb, PB, prestaged);
}
// the single-group staging of backsub_warp, callable ahead of time (factor columns [base, top) -> Bw, reciprocal pivots behind them)
__device__ void backsub_stage(const double* __restrict__ Lb_g, double* Bw, int base, int top, int kd, int ldb, int PB) {
  const int tid = threadIdx.x, nt = blockDim.x, total = (top - base) * ldb;
  const double* src = Lb_g + (int64_t)base * ldb;
  double* ipv = Bw + (size_t)(PB + kd) * ldb;
  for (int b0 = tid; b0 < total; b0 += 8 * nt) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) { const int idx = b0 + u * nt; v[u] = idx < total ? src[idx] : 0.0; }
#pragma unroll
    for (int u = 0; u < 8; ++u) { const int idx = b0 + u * nt; if (idx < total) Bw[idx] = v[u]; }
  }
  for (int idx = tid; idx < top - base; idx += nt) ipv[idx] = 1.0 / Lb_g[(int64_t)(base + idx) * ldb];
}

// shared-memory carve-up shared by kernels A and B
__device__ FactorSmem carve_smem(double* sm, int WS, int CL, int nbl, int kd, int ldbp, double** extra, int extra_doubles, double* cl_ext = nullptr) {
  FactorSmem fs;
  fs.W = sm;
  double* p = fs.W + (size_t)WS * CL;
  if (cl_ext) fs.Cl = cl_ext; else { fs.Cl = p; p += nbl * nbl; }
  *extra = p; p += extra_doubles;
  fs.inv = p; p += 2 * KB;
  fs.Ld = p; p += 2 * KB * KB;
  fs.nbl = nbl;
  fs.flag = reinterpret_cast<int*>(p);
  fs.blocks = reinterpret_cast<uchar2*>(fs.flag + 2);
  fs.nblocks = 0;
  return fs;
}
__host__ __device__ inline size_t factor_smem_bytes(int WS, int CL, int nbl, int kd, int extra_doubles, bool cl_in_smem = true) {
  const int nbk = (kd + nbl + 7) / 8;
  return ((size_t)WS * CL + (cl_in_smem ? (size_t)nbl * nbl : 0) + extra_doubles + 2 * KB + 2 * KB * KB + 1) * sizeof(double) + (size_t)nbk * (nbk + 1) / 2 * sizeof(uchar2) + 64;
}

// ---- dense front elimination (cyclic-reduction levels and the root) ------------------------------------------------
// A front is the dense column panel of one separator block: rows [own block (w) | trailing rows (mt)], columns = the w pivots,
// column-major in shared memory with zero padding (rows to a multiple of 8 past the own block, columns to a multiple of 4),
// unscaled storage as in the band factor (diagonal = D_j, below = L_ij D_j).  The panel is factored in sub-panels of KB
// columns (one lane factors the KB x KB block in registers, PWD warps substitute the rows below, all warps apply the rank-KB
// update to the remaining panel columns on the tensor cores); the Schur complement of the trailing rows is then formed in ONE
// pass with register accumulators over all w pivots and handed, entry by entry, to a sink (atomics into the next level / the
// root's border block).
constexpr int PWD = 4;
struct DenseFront { double* Pn; int ld, w, mt, MF, rows; double* inv; double* Ld; int* flag; };   // MF = w + mt, rows = allocated (padded) rows
__host__ __device__ inline int front_rows(int w, int mt) { return w + ((mt + 7) & ~7); }
__host__ __device__ inline int front_ld(int w, int mt) { return front_rows(w, mt) | 1; }
__host__ __device__ inline int front_cols(int w) { return (w + KB - 1) / KB * KB; }
__host__ __device__ inline size_t front_doubles(int w, int mt) { return (size_t)front_ld(w, mt) * front_cols(w) + front_cols(w) + KB * KB + 2; }
__device__ DenseFront carve_front(double* sm, int w, int mt) {
  DenseFront f; f.Pn = sm; f.w = w; f.mt = mt; f.MF = w + mt; f.rows = front_rows(w, mt); f.ld = front_ld(w, mt);
  f.inv = f.Pn + (size_t)f.ld * front_cols(w); f.Ld = f.inv + front_cols(w); f.flag = reinterpret_cast<int*>(f.Ld + KB * KB);
  return f;
}

// KB x KB diagonal block of a sub-panel, factored by ONE thread in registers (its own function: the 36 + 8 live doubles must not
// compete with the caller's registers under the 128-register cap of a 512-thread CTA)
__device__ __noinline__ void dense_block_factor(double* Pn, int ld, int j0, int kb, double* inv, double* Ld, int* flag) {
  double a[KB][KB];
  double* p0 = Pn + (size_t)j0 * ld + j0;
#pragma unroll
  for (int c = 0; c < KB; ++c)
#pragma unroll
    for (int r = 0; r < KB; ++r) if (r >= c) a[r][c] = p0[(size_t)c * ld + r];   // padding columns / rows are zero
  bool ok = true;
  // constant-trip loops with compile-time predicates only: the triangular loop nest otherwise leaves a[][] in local memory;
  // column j is final once pivot j is known, so it is written back at once (keeps the live register set shrinking)
#pragma unroll
  for (int j = 0; j < KB; ++j) {
    const double D = a[j][j];
    const bool piv = j < kb;                                      // columns past the block end are no pivots: iv = 0 makes them inert
    if (piv && (!(D > 0.0) || !isfinite(D))) ok = false;
    const double iv = piv ? 1.0 / D : 0.0;
#pragma unroll
    for (int c = 0; c < KB; ++c) {
      if (c > j) {
        const double lcj = a[c][j] * iv;
        Ld[c * KB + j] = lcj;
#pragma unroll
        for (int i = 0; i < KB; ++i) if (i >= c) a[i][c] = fma(-a[i][j], lcj, a[i][c]);
      }
    }
    if (piv) {
      inv[j0 + j] = iv;
#pragma unroll
      for (int r = 0; r < KB; ++r) if (r >= j) p0[(size_t)j * ld + r] = a[r][j];
    }
  }
  if (!ok) *flag = 0;
}

__device__ __forceinline__ void dense_subpanel_factor(const DenseFront& f, int j0, int kb) {   // warps 0..PWD-1
  const int gl = threadIdx.x, ld = f.ld;
  double* Pn = f.Pn; double* Ld = f.Ld;
  if (gl == 0) dense_block_factor(Pn, ld, j0, kb, f.inv, Ld, f.flag);
  asm volatile("bar.sync 1, %0;" :: "r"(PWD * 32) : "memory");
  double lreg[KB * (KB - 1) / 2];
  {
    int q = 0;
#pragma unroll
    for (int c = 1; c < KB; ++c)
#pragma unroll
      for (int k = 0; k < c; ++k) lreg[q++] = Ld[c * KB + k];
  }
  for (int x = j0 + KB + gl; x < f.MF; x += PWD * 32) {
    double wv[KB];
#pragma unroll
    for (int c = 0; c < KB; ++c) wv[c] = c < kb ? Pn[(size_t)(j0 + c) * ld + x] : 0.0;
    int q = 0;
#pragma unroll
    for (int c = 1; c < KB; ++c) {
      double v = wv[c];
#pragma unroll
      for (int k = 0; k < c; ++k) v = fma(-wv[k], lreg[q++], v);
      wv[c] = v;
      if (c < kb) Pn[(size_t)(j0 + c) * ld + x] = v;
    }
  }
}

// rank-KB update of the panel columns [c_begin, c_end) (c_begin = j0 + KB + multiple of 8) with the finished sub-panel at j0
__device__ __forceinline__ void dense_panel_update(const DenseFront& f, int j0, int c_begin, int c_end, int wslot, int nslots) {
  const int lane = threadIdx.x & 31, fr = lane >> 2, fk = lane & 3, ld = f.ld;
  double* Pn = f.Pn;
  int idx = wslot;
  for (int cs = c_begin; cs < c_end; cs += 8) {
    const int nbr = (f.MF - cs + 7) / 8;                         // block rows from the diagonal block of this block column down
    for (; idx < nbr; idx += nslots) {
      const int xa = cs + 8 * idx + fr;                          // < f.rows (padding rows are zero)
      double acc[2] = {0.0, 0.0};
#pragma unroll
      for (int ks = 0; ks < KB / 4; ++ks) {
        const int jj = j0 + 4 * ks + fk;
        const double* cj = Pn + (size_t)jj * ld;
        dmma_acc(acc, -cj[xa] * f.inv[jj], cj[cs + fr]);
      }
#pragma unroll
      for (int e = 0; e < 2; ++e) { const int y = cs + 2 * fk + e; if (y < f.w && xa >= y && xa < f.MF) Pn[(size_t)y * ld + xa] += acc[e]; }
    }
    idx -= nbr;
  }
}

// sub-panel loop with a look-ahead of depth one: the next sub-panel's columns are updated first, then PWD warps factor it while
// the other warps finish the update of the remaining panel columns
__device__ bool dense_front_factor(const DenseFront& f) {
  const int warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5, w = f.w;
  if (warp < PWD) dense_subpanel_factor(f, 0, min(KB, w));
  __syncthreads();
  if (*f.flag == 0) return false;
  for (int j0 = 0; j0 + KB < w; j0 += KB) {
    dense_panel_update(f, j0, j0 + KB, min(j0 + 2 * KB, w), warp, nwarps);
    __syncthreads();
    if (warp < PWD) dense_subpanel_factor(f, j0 + KB, min(KB, w - j0 - KB));
    else dense_panel_update(f, j0, j0 + 2 * KB, w, warp - PWD, nwarps - PWD);
    __syncthreads();
    if (*f.flag == 0) return false;
  }
  return true;
}

// Schur complement of the trailing rows: sink(x, y, v) receives v = -sum_j L_xj D_j L_yj for mt > x >= y >= 0
template <class Sink>
__device__ __forceinline__ void dense_front_schur(const DenseFront& f, Sink sink) {
  const int lane = threadIdx.x & 31, fr = lane >> 2, fk = lane & 3, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5, ld = f.ld;
  const int nbt = (f.mt + 7) / 8, nblk = nbt * (nbt + 1) / 2, ksteps = (f.w + 3) / 4;
  const double* T = f.Pn + f.w;                                  // trailing rows of every column
  for (int b = warp; b < nblk; b += nwarps) {
    const int bi = tri_row(b), bj = b - bi * (bi + 1) / 2;
    const int xa = 8 * bi + fr, xb = 8 * bj + fr;
    // three independent accumulator chains; columns >= w are zero padding with inv = 0
    double acc[2] = {0.0, 0.0}, acc1[2] = {0.0, 0.0}, acc2[2] = {0.0, 0.0};
    const double* cj = T + (size_t)fk * ld;
    const double* iv = f.inv + fk;
    int ks = 0;
    for (; ks + 3 <= ksteps; ks += 3, cj += 12 * (size_t)ld, iv += 12) {
      const double a0 = cj[xa], b0 = cj[xb], i0 = iv[0];
      const double a1 = cj[4 * (size_t)ld + xa], b1 = cj[4 * (size_t)ld + xb], i1 = iv[4];
      const double a2 = cj[8 * (size_t)ld + xa], b2 = cj[8 * (size_t)ld + xb], i2 = iv[8];
      dmma_acc(acc, -a0 * i0, b0); dmma_acc(acc1, -a1 * i1, b1); dmma_acc(acc2, -a2 * i2, b2);
    }
    for (; ks < ksteps; ++ks, cj += 4 * (size_t)ld, iv += 4) dmma_acc(acc, -cj[xa] * iv[0], cj[xb]);
    acc[0] += acc1[0] + acc2[0]; acc[1] += acc1[1] + acc2[1];
#pragma unroll
    for (int e = 0; e < 2; ++e) { const int y = 8 * bj + 2 * fk + e; if (xa >= y && xa < f.mt) sink(xa, y, acc[e]); }
  }
}

// factor columns -> global factor storage shared with the band back-substitution: Lb[col][e] (e = 0: pivot; own rows, then
// the right block) and El[col][left | border | rhs]; trailing row order of a front: [left (wl) | right (wr) | border + rhs]
__device__ void dense_front_store(const DenseFront& f, int wl, int wr, int nbp, double* Lb, int ldb, int kd, double* El, int nbl) {
  const int w = f.w, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int j = warp; j < w; j += nwarps) {
    const double* cj = f.Pn + (size_t)j * f.ld;
    for (int e = lane; e <= kd; e += 32) { const int r = j + e; Lb[(int64_t)j * ldb + e] = r < w ? cj[r] : (r - w < wr ? cj[w + wl + (r - w)] : 0.0); }
    for (int i = lane; i < nbl; i += 32) El[(int64_t)j * nbl + i] = i < w ? (i < wl ? cj[w + i] : 0.0) : cj[w + wl + wr + (i - w)];
  }
}

// ---- kernel A0: materialise the scaled + damped window columns of every chunk (fully parallel) ----------------------
// Wg[col][e]: e < ldbp band entries (zero padding beyond kd, rows beyond the chunk's right separator masked), then the local
// border [coupling to the left separator (stored transposed in H) | border | rhs].  Kernel A then only copies columns.
__global__ void prepare_kernel(DeviceProblem P, SolvePlan pl, const double* __restrict__ scale, SolveParams sp, double* wsp, double* scal) {
  const int c = blockIdx.x, nk = P.nk, nb = P.nb, kd = P.kd, ldb = P.ldb, w = pl.w, nbl = pl.nbl;
  const int a = chunk_a(pl, c), b = chunk_b(pl, c);
  const bool has_left = c > 0, has_right = c < pl.P - 1;
  const int ldbp = kd + KB, CL = ldbp + nbl, right_end = has_right ? b + w : b;
  const double* band = P.ne; const double* E = P.ne + P.ne_off_E; const double* g = P.ne + P.ne_off_g;
  SolveWs ws = carve(wsp, nk, nb, ldb, pl);
  pdl_wait_then_trigger();
  if (scal && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < 5) scal[threadIdx.x] = 0.0;   // model change, step / x norms, candidate cost, ok
  const int total = (right_end - a) * CL, stride = gridDim.y * blockDim.x, de = stride % CL, dc = stride / CL;
  const int idx0 = blockIdx.y * blockDim.x + threadIdx.x;
  int e = idx0 % CL, col = a + idx0 / CL;
  for (int idx = idx0; idx < total; idx += stride, e += de, col += dc) {
    if (e >= CL) { e -= CL; ++col; }
    double v = 0.0;
    if (e < ldbp) {
      const int i = col + e;
      if (e <= kd && i < nk && i < right_end) { v = band[(int64_t)col * ldb + e] * scale[col] * scale[i]; if (e == 0) v += lm_d2(P, scale, sp, col); }
    } else {
      const int lb = e - ldbp;
      if (lb < w) { if (has_left && col < b) { const int s = a - w + lb, off = col - s; if (off <= kd) v = band[(int64_t)s * ldb + off] * scale[s] * scale[col]; } }
      else if (lb < w + nb) v = E[(int64_t)col * nb + (lb - w)] * scale[col] * scale[nk + lb - w];
      else v = -g[col] * scale[col];
    }
    ws.Wg[(int64_t)col * CL + e] = v;
  }
}

// ---- level 0: eliminate the interior knots of every time chunk ----------------------------------------------------
__global__ void __launch_bounds__(NT) eliminate_kernel(DeviceProblem P, SolvePlan pl, double* wsp, double* scal) {
  extern __shared__ __align__(16) double sm[];
  const int c = blockIdx.x, nk = P.nk, nb = P.nb, w = pl.w, nbl = pl.nbl, nbp = nb + 1, kd = P.kd, ldb = P.ldb;
  SolveWs ws = carve(wsp, nk, nb, P.ldb, pl);
  const int a = chunk_a(pl, c), b = chunk_b(pl, c);
  const bool has_left = c > 0, has_right = c < pl.P - 1;
  const int ldbp = kd + KB, CL = ldbp + nbl, WS = pl.WS_A;
  double* extra;
  FactorSmem fs = carve_smem(sm, WS, CL, nbl, kd, ldbp, &extra, 0, pl.cl_global ? ws.Clg + (size_t)c * nbl * nbl : nullptr);
  double* W = fs.W; double* Cl = fs.Cl;
  fs.nblocks = build_block_table(fs.blocks, kd + nbl);
  for (int i = threadIdx.x; i < nbl * nbl; i += blockDim.x) Cl[i] = 0.0;
  pdl_wait_then_trigger();
  __syncthreads();
  const int right_end = has_right ? b + w : b;
  auto load = [&](int col, int e) -> double { return col < right_end ? ws.Wg[(int64_t)col * CL + e] : 0.0; };
  auto store = [&](int col, int e, double v) { if (e < ldbp) { if (e <= kd) ws.Lb[(int64_t)col * ldb + e] = v; } else ws.El[(int64_t)col * nbl + (e - ldbp)] = v; };
  const bool ok = factor_range(fs, a, b, kd, ldbp, CL, WS, load, store);
  if (!ok) { if (threadIdx.x == 0) scal[SC_OK] = -1.0; return; }
  // ---- scatter the Schur complement into the first reduced system: the left / right separators are its blocks c-1 / c ----
  const int mask = WS - 1;
  const int sl0 = (c - 1) * w, sr0 = c * w;
  double* ob = ws.bandr; double* oE = ws.Er;
  if (has_right) {
    for (int idx = threadIdx.x; idx < w * CL; idx += blockDim.x) {
      const int t = idx / CL, e = idx % CL, col = b + t;
      const double v = W[(size_t)(col & mask) * CL + e];
      if (v == 0.0) continue;
      if (e < ldbp) { if (t + e < w) atomicAdd(ob + (int64_t)(sr0 + t) * pl.ldbr + e, v); }
      else {
        const int lb = e - ldbp;
        if (lb < w) { if (has_left) atomicAdd(ob + (int64_t)(sl0 + lb) * pl.ldbr + (sr0 + t - sl0 - lb), v); }
        else atomicAdd(oE + (int64_t)(sr0 + t) * nbp + (lb - w), v);
      }
    }
  }
  for (int idx = threadIdx.x; idx < nbl * (nbl + 1) / 2; idx += blockDim.x) {
    const int b1 = tri_row(idx), b2 = idx - b1 * (b1 + 1) / 2;   // b1 >= b2, local order [left | border | rhs]
    const double v = Cl[b1 * nbl + b2];
    if (v == 0.0) continue;
    if (b1 < w) { if (has_left) atomicAdd(ob + (int64_t)(sl0 + b2) * pl.ldbr + (b1 - b2), v); }
    else if (b2 < w) { if (has_left) atomicAdd(oE + (int64_t)(sl0 + b2) * nbp + (b1 - w), v); }
    else atomicAdd(ws.Cr + (int64_t)(b1 - w) * nbp + (b2 - w), v);
  }
}

// ---- level l >= 1: cyclic reduction -- eliminate every other block of the block-tridiagonal system R_l ------------------
// CTA c eliminates block 2c; its neighbours 2c-1 / 2c+1 become blocks c-1 / c of R_{l+1}.  Front rows: [own | left | right | border | rhs].
__global__ void __launch_bounds__(NT) reduce_kernel(DeviceProblem P, SolvePlan pl, int level, double* wsp, double* scal) {
  extern __shared__ __align__(16) double sm[];
  const int c = blockIdx.x, nk = P.nk, nb = P.nb, w = pl.w, nbl = pl.nbl, nbp = nb + 1, ldb = pl.ldbr, kd = pl.kdr;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
  SolveWs ws = carve(wsp, nk, nb, P.ldb, pl);
  const int o = pl.off[level], a = 2 * c * w, b = a + w;
  const bool has_left = c > 0, has_right = 2 * c + 1 < pl.S[level];
  const double* src_band = ws.bandr + (int64_t)o * ldb; const double* src_E = ws.Er + (int64_t)o * nbp;
  double* ob = ws.bandr + (int64_t)pl.off[level + 1] * ldb; double* oE = ws.Er + (int64_t)pl.off[level + 1] * nbp;
  const int mt = 2 * w + nbp;
  DenseFront f = carve_front(sm, w, mt);
  for (int i = tid; i < (int)front_doubles(w, mt) - 2; i += nt) f.Pn[i] = 0.0;   // panel (with padding), inv, Ld
  if (tid == 0) *f.flag = 1;
  pdl_wait_then_trigger();
  if (scal[SC_OK] < 0.0) return;                                 // an earlier level hit a bad pivot (uniform)
  __syncthreads();
  const int sl0 = (c - 1) * w, sr0 = c * w;
  auto fetch = [&](int j, int r) -> double {                     // entry (row r, pivot column j) of the front
    if (r >= f.MF) return 0.0;
    const double* bj = src_band + (int64_t)(a + j) * ldb;
    if (r < w) return r >= j ? bj[r - j] : 0.0;
    if (r < 2 * w) { const int lb = r - w; return has_left ? src_band[(int64_t)(a - w + lb) * ldb + (w + j - lb)] : 0.0; }
    if (r < 3 * w) return has_right ? bj[r - w - j] : 0.0;       // row b + (r - 2w): offset w + (r - 2w) - j
    return src_E[(int64_t)(a + j) * nbp + (r - 3 * w)];
  };
  {   // gather the front: (column, 32-row chunk) items dealt round-robin to the warps, 8 independent loads per lane in flight
    const int chunks = (f.MF + 31) >> 5, items = w * chunks;
    for (int it0 = warp; it0 < items; it0 += 8 * nwarps) {
      double v[8]; int dst[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int it = it0 + u * nwarps;
        dst[u] = -1; v[u] = 0.0;
        if (it < items) { const int j = it / chunks, r = ((it - j * chunks) << 5) + lane; if (r < f.MF) { v[u] = fetch(j, r); dst[u] = j * f.ld + r; } }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) if (dst[u] >= 0) f.Pn[dst[u]] = v[u];
    }
  }
  if (has_right) {                                               // the right neighbour carries its own entries to the next level
    const int rw = w + nbp, tot = w * rw;
    for (int base = tid; base < tot; base += 4 * nt) {
      double v[4]; double* dst[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = base + u * nt; v[u] = 0.0; dst[u] = nullptr;
        if (idx < tot) {
          const int t = idx / rw, e = idx % rw;
          if (e < w) { if (t + e < w) { v[u] = src_band[(int64_t)(b + t) * ldb + e]; dst[u] = ob + (int64_t)(sr0 + t) * ldb + e; } }
          else { v[u] = src_E[(int64_t)(b + t) * nbp + (e - w)]; dst[u] = oE + (int64_t)(sr0 + t) * nbp + (e - w); }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) if (dst[u] && v[u] != 0.0) atomicAdd(dst[u], v[u]);
    }
  }
  __syncthreads();
  if (!dense_front_factor(f)) { if (tid == 0) scal[SC_OK] = -1.0; return; }
  dense_front_store(f, w, w, nbp, ws.Lbr + (int64_t)(o + a) * ldb, ldb, kd, ws.Elr + (int64_t)(o + a) * nbl, nbl);
  dense_front_schur(f, [&](int x, int y, double v) {             // trailing order [left | right | border | rhs], x >= y
    if (y < w) {
      if (!has_left) return;
      if (x < w) atomicAdd(ob + (int64_t)(sl0 + y) * ldb + (x - y), v);
      else if (x < 2 * w) { if (has_right) atomicAdd(ob + (int64_t)(sl0 + y) * ldb + (sr0 + (x - w) - sl0 - y), v); }
      else atomicAdd(oE + (int64_t)(sl0 + y) * nbp + (x - 2 * w), v);
    } else if (y < 2 * w) {
      if (!has_right) return;
      if (x < 2 * w) atomicAdd(ob + (int64_t)(sr0 + y - w) * ldb + (x - y), v);
      else atomicAdd(oE + (int64_t)(sr0 + y - w) * nbp + (x - 2 * w), v);
    } else atomicAdd(ws.Cr + (int64_t)(x - 2 * w) * nbp + (y - 2 * w), v);
  });
}

// ---- root: last separator block (if any) + border: factor, solve ------------------------------------------------------
__global__ void __launch_bounds__(NT) root_kernel(DeviceProblem P, SolvePlan pl, const double* __restrict__ scale, SolveParams sp, double* wsp, double* scal) {
  extern __shared__ __align__(16) double sm[];
  const int nk = P.nk, nb = P.nb, nbp = nb + 1, root = pl.L + 1, nkr = pl.S[root] * pl.w, kdr = pl.kdr, ldbr = pl.ldbr, w = pl.w, nbl = pl.nbl;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
  // nbp x nbp lower, row nb = rhs; wide borders keep it in HBM (L2 resident)
  double* xb = pl.cs_global ? sm : sm + nbp * nbp;   // border solution
  double* rest = xb + ((nbp + 4) & ~3);            // dense front, later the back-substitution staging
  const double* C = P.ne + P.ne_off_C; const double* g = P.ne + P.ne_off_g;
  SolveWs ws = carve(wsp, nk, nb, P.ldb, pl);
  double* Cs = pl.cs_global ? ws.Csg : sm;
  const double* rband = ws.bandr + (int64_t)pl.off[root] * ldbr; const double* rE = ws.Er + (int64_t)pl.off[root] * nbp;
  double* rLb = ws.Lbr + (int64_t)pl.off[root] * ldbr; double* rEl = ws.Elr + (int64_t)pl.off[root] * nbl;
  pdl_wait_then_trigger();
  if (scal[SC_OK] < 0.0) { if (tid == 0) { scal[SC_OK] = 0.0; scal[SC_MODEL_CHANGE] = 0.0; } return; }   // an elimination hit a bad pivot
  for (int idx = tid; idx < nbp * nbp; idx += nt) {
    const int b = idx / nbp, c = idx % nbp;
    double v = 0.0;
    if (c <= b) {
      v = ws.Cr[idx];                                                       // Schur contributions of all levels
      if (b < nb) { v += C[(int64_t)b * nb + c] * scale[nk + b] * scale[nk + c]; if (b == c) v += lm_d2(P, scale, sp, nk + b); }
      else if (c < nb) v += -g[nk + c] * scale[nk + c];
    }
    Cs[idx] = v;
  }
  bool ok = true;
  if (nkr > 0) {                                   // one remaining block: front rows [own | border | rhs]
    DenseFront f = carve_front(rest, w, nbp);
    for (int i = tid; i < (int)front_doubles(w, nbp) - 2; i += nt) f.Pn[i] = 0.0;
    if (tid == 0) *f.flag = 1;
    __syncthreads();
    for (int j = warp; j < w; j += nwarps) {
      double* cj = f.Pn + (size_t)j * f.ld;
      for (int r = lane; r < f.MF; r += 32) cj[r] = r < w ? (r >= j ? rband[(int64_t)j * ldbr + (r - j)] : 0.0) : rE[(int64_t)j * nbp + (r - w)];
    }
    __syncthreads();
    ok = dense_front_factor(f);
    if (ok) {
      dense_front_store(f, 0, 0, nbp, rLb, ldbr, kdr, rEl, nbl);
      dense_front_schur(f, [&](int x, int y, double v) { Cs[x * nbp + y] += v; });
    }
  }
  __syncthreads();
  // border: dense LDL^T of the final Schur complement, rhs carried as the last row
  for (int j = 0; j < nb && ok; ++j) {
    const double piv = Cs[j * nbp + j];
    if (!(piv > 0.0) || !isfinite(piv)) { ok = false; break; }
    const double inv = 1.0 / piv;
    const int mrem = nbp - 1 - j;
    for (int idx = tid; idx < mrem * (mrem + 1) / 2; idx += nt) {
      const int r = tri_row(idx), c = idx - r * (r + 1) / 2;
      const int b = j + 1 + r, cc = j + 1 + c;
      Cs[b * nbp + cc] -= Cs[b * nbp + j] * Cs[cc * nbp + j] * inv;
    }
    __syncthreads();
  }
  if (!ok) { if (tid == 0) { scal[SC_OK] = 0.0; scal[SC_MODEL_CHANGE] = 0.0; } return; }
  if (tid < 32) {   // border back-substitution
    for (int b = tid; b < nb; b += 32) xb[b] = Cs[nb * nbp + b];
    __syncwarp();
    for (int j = nb - 1; j >= 0; --j) {
      const double xj = xb[j] / Cs[j * nbp + j];
      __syncwarp();
      if (tid == 0) xb[j] = xj;
      for (int i = tid; i < j; i += 32) xb[i] -= Cs[j * nbp + i] * xj;
      __syncwarp();
    }
  }
  __syncthreads();
  for (int b = tid; b < nb; b += nt) ws.y[nk + b] = xb[b];
  if (nkr > 0) {
    // remaining block: t_j = rhs_j - sum_b El[j][border b] x_b, then the register/shuffle back-substitution
    double* tw = rest; double* Bw = rest + ((nkr + 3) & ~3);
    for (int j = tid; j < nkr; j += nt) { const double* le = rEl + (int64_t)j * nbl + w; double t = le[nb]; for (int b = 0; b < nb; ++b) t -= le[b] * xb[b]; tw[j] = t; }
    __syncthreads();
    backsub_dispatch(rLb, tw, Bw, 0, nkr, nkr, kdr, ldbr, 64);
    for (int rj = tid; rj < nkr; rj += nt) ws.y[sep_col(pl, root, 0) + rj] = tw[rj];
  }
  __syncthreads();
  if (tid == 0) scal[SC_OK] = 1.0;
}

// ---- back-substitution of one level (level 0: chunk interiors, level >= 1: the blocks eliminated at that level) -----
template <bool LEVEL0>
__global__ void __launch_bounds__(NT) backsub_kernel(DeviceProblem P, SolvePlan pl, int level, double* wsp, const double* scal) {
  extern __shared__ __align__(16) double sm[];
  const int c = blockIdx.x, nk = P.nk, nb = P.nb, w = pl.w, nbl = pl.nbl, tid = threadIdx.x, nt = blockDim.x;
  SolveWs ws = carve(wsp, nk, nb, P.ldb, pl);
  int a, b, kd, ldb, y_left, y_own, y_right; bool has_left, has_right;   // y_*: position of the blocks in the solution vector
  const double* Lb; const double* El;
  if (LEVEL0) {
    a = chunk_a(pl, c); b = chunk_b(pl, c); kd = P.kd; ldb = P.ldb; has_left = c > 0; has_right = c < pl.P - 1;
    Lb = ws.Lb; El = ws.El; y_left = a - w; y_own = a; y_right = b;
  } else {
    const int o = pl.off[level];
    a = 2 * c * w; b = a + w; kd = pl.kdr; ldb = pl.ldbr; has_left = c > 0; has_right = 2 * c + 1 < pl.S[level];
    Lb = ws.Lbr + (int64_t)o * ldb; El = ws.Elr + (int64_t)o * nbl;
    y_left = has_left ? sep_col(pl, level, 2 * c - 1) : 0; y_own = sep_col(pl, level, 2 * c); y_right = has_right ? sep_col(pl, level, 2 * c + 1) : 0;
  }
  const int top = has_right ? b + w : b;   // right separator values are known: they only enter the right-hand sides
  const int PB = LEVEL0 ? 128 : 64;
  const bool staged = b - a <= PB && (!LEVEL0 || pl.stage0);   // the usual case: the factor of this block is staged BEFORE waiting for the predecessor
  double* xl = sm;                         // local border solution [left separator | border]
  double* xr = xl + ((nbl + 3) & ~3);      // right separator solution
  double* tw = xr + ((w + 3) & ~3);        // t / x for columns [a, b)
  double* Bw = tw + ((b - a + 3) & ~3);    // (PB + kd) * ldb panel of L, then PB reciprocal pivots
  double* Els = Bw + (size_t)(PB + kd) * ldb + PB;   // staged rows of El
  if (staged) {   // written by the elimination kernels, i.e. older than the direct predecessor: safe before the wait
    backsub_stage(Lb, Bw, a, b, kd, ldb, PB);
    const double* src = El + (int64_t)a * nbl;
    for (int i = tid; i < (b - a) * nbl; i += nt) Els[i] = src[i];
  }
  pdl_wait_then_trigger();
  if (scal[SC_OK] != 1.0) return;
  for (int i = tid; i < w + nb; i += nt) xl[i] = i < w ? (has_left ? ws.y[y_left + i] : 0.0) : ws.y[nk + i - w];
  for (int i = tid; i < w; i += nt) xr[i] = has_right ? ws.y[y_right + i] : 0.0;
  __syncthreads();
  // t_j = rhs_j - sum_i El[j][i] xl[i] - sum_{r in right separator} (L_rj D_j) x_r : one warp per column
  const int lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
  for (int j = a + warp; j < b; j += nwarps) {
    const double* le = staged ? Els + (size_t)(j - a) * nbl : El + (int64_t)j * nbl;
    const double* lc = staged ? Bw + (size_t)(j - a) * ldb : Lb + (int64_t)j * ldb;
    double acc = 0.0;
    for (int i = lane; i < w + nb; i += 32) acc = fma(le[i], xl[i], acc);
    for (int r = b + lane; r < top && r - j <= kd; r += 32) acc = fma(lc[r - j], xr[r - b], acc);
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) tw[j - a] = le[w + nb] - acc;
  }
  __syncthreads();
  backsub_dispatch(Lb, tw, Bw, a, b, b, kd, ldb, PB, staged);
  for (int j = a + tid; j < b; j += nt) ws.y[y_own + (j - a)] = tw[j - a];
}

// ---- kernel D: step in the unscaled space, model cost change = 1/2 (y^T D y + y^T rhs) ----------------------------
__global__ void finish_kernel(DeviceProblem P, SolvePlan pl, const double* __restrict__ scale, SolveParams sp, double* wsp, double* delta, double* scal) {
  pdl_wait_then_trigger();
  if (scal[SC_OK] != 1.0) return;
  const int n = P.nk + P.nb;
  SolveWs ws = carve(wsp, P.nk, P.nb, P.ldb, pl);
  const double* g = P.ne + P.ne_off_g;
  double part = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double yi = ws.y[i], s = scale[i];
    delta[i] = yi * s;
    part += lm_d2(P, scale, sp, i) * yi * yi - yi * g[i] * s;
  }
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(scal + SC_MODEL_CHANGE, 0.5 * part);
}

__global__ void scale_kernel(DeviceProblem P, double* scale, int jacobi, double* scal) {
  const int n = P.nk + P.nb;
  __shared__ double red[32];
  double gmax = 0.0;
  const double* g = P.ne + P.ne_off_g;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double d = i < P.nk ? P.ne[(int64_t)i * P.ldb] : P.ne[P.ne_off_C + (int64_t)(i - P.nk) * P.nb + (i - P.nk)];
    if (scale) scale[i] = jacobi ? 1.0 / (1.0 + sqrt(d)) : 1.0;
    gmax = fmax(gmax, fabs(g[i]));
  }
  for (int o = 16; o > 0; o >>= 1) gmax = fmax(gmax, __shfl_xor_sync(0xffffffffu, gmax, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = gmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = 0.0;
    for (int w = 0; w < (blockDim.x + 31) / 32; ++w) m = fmax(m, red[w]);
    atomicMax(reinterpret_cast<unsigned long long*>(scal + SC_GRAD_MAX), (unsigned long long)__double_as_longlong(m));   // non-negative doubles order like their bits
    if (blockIdx.x == 0) scal[SC_X_COST] = P.ne[P.ne_off_cost];   // cost at the linearisation point, read back with the step scalars
  }
}

// SE3::exp (sophus/se3.hpp:761-783), tangent = (upsilon, omega)
__device__ void se3_exp_dev(const double* a, Q4& q, V3& t) {
  const V3 ups = v3(a[0], a[1], a[2]), om = v3(a[3], a[4], a[5]);
  const double th2 = dot(om, om);
  const ExpOut e = so3_exp_jr(om);
  q = e.q;
  if (th2 < kEps * kEps) { t = qrot(q, ups); return; }   // V = so3.matrix() branch
  const V3 c1 = cross(om, ups);                          // V = I + (1-cos t)/t^2 [om]x + (t - sin t)/t^3 [om]x^2
  t = ups + e.a * c1 + e.b * cross(om, c1);
}

__global__ void update_kernel(DeviceProblem P, DeviceState cur, DeviceState cand, const double* __restrict__ delta, double max_ba, double max_bg, double* scal) {
  pdl_wait_then_trigger();
  const int total = P.n_so3 + P.n_r3 + P.n_ba + P.n_bg + 1;
  double step = 0.0, xsq = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    if (i < P.n_so3) {
      const double4 k = cur.so3[i];
      const int c = P.so3_col[i];
      double4 o = k;
      if (c >= 0) {
        const Q4 r = qnormalized(qmul(q4(k.x, k.y, k.z, k.w), so3_exp(v3(delta[c], delta[c + 1], delta[c + 2]))));
        o = make_double4(r.x, r.y, r.z, r.w);
        step += (o.x - k.x) * (o.x - k.x) + (o.y - k.y) * (o.y - k.y) + (o.z - k.z) * (o.z - k.z) + (o.w - k.w) * (o.w - k.w);
        xsq += k.x * k.x + k.y * k.y + k.z * k.z + k.w * k.w;
      }
      cand.so3[i] = o;
    } else if (i < P.n_so3 + P.n_r3) {
      const int j = i - P.n_so3;
      const double4 k = cur.r3[j];
      const int c = P.r3_col[j];
      double4 o = k;
      if (c >= 0) {
        o = make_double4(k.x + delta[c], k.y + delta[c + 1], k.z + delta[c + 2], 0.0);
        step += (o.x - k.x) * (o.x - k.x) + (o.y - k.y) * (o.y - k.y) + (o.z - k.z) * (o.z - k.z);
        xsq += k.x * k.x + k.y * k.y + k.z * k.z;
      }
      cand.r3[j] = o;
    } else if (i < P.n_so3 + P.n_r3 + P.n_ba + P.n_bg) {
      const bool is_a = i < P.n_so3 + P.n_r3 + P.n_ba;
      const int j = is_a ? i - P.n_so3 - P.n_r3 : i - P.n_so3 - P.n_r3 - P.n_ba;
      const double4 k = is_a ? cur.ba[j] : cur.bg[j];
      const int c = is_a ? P.ba_col[j] : P.bg_col[j];
      const double lim = is_a ? max_ba : max_bg;
      double4 o = k;
      if (c >= 0) {   // box constraints of SetFixedParams (impl.h:206-251), enforced by projection
        o = make_double4(fmin(fmax(k.x + delta[c], -lim), lim), fmin(fmax(k.y + delta[c + 1], -lim), lim), fmin(fmax(k.z + delta[c + 2], -lim), lim), 0.0);
        step += (o.x - k.x) * (o.x - k.x) + (o.y - k.y) * (o.y - k.y) + (o.z - k.z) * (o.z - k.z);
        xsq += k.x * k.x + k.y * k.y + k.z * k.z;
      }
      if (is_a) cand.ba[j] = o; else cand.bg[j] = o;
    } else {
      double gl[G_COUNT];
      for (int k = 0; k < G_COUNT; ++k) gl[k] = cur.glob[k];
      if (P.col_tic >= 0) {
        Q4 dq; V3 dt;
        se3_exp_dev(delta + P.col_tic, dq, dt);
        const Q4 q = q4(gl[0], gl[1], gl[2], gl[3]);
        const Q4 r = qnormalized(qmul(q, dq));
        const V3 t = v3(gl[4], gl[5], gl[6]) + qrot(q, dt);
        const double nv[7] = {r.x, r.y, r.z, r.w, t.x, t.y, t.z};
        for (int k = 0; k < 7; ++k) { step += (nv[k] - gl[k]) * (nv[k] - gl[k]); xsq += gl[k] * gl[k]; gl[k] = nv[k]; }
      }
      if (P.col_g >= 0) for (int k = 0; k < 3; ++k) { const double d = delta[P.col_g + k]; step += d * d; xsq += gl[G_GRAV + k] * gl[G_GRAV + k]; gl[G_GRAV + k] += d; }
      if (P.col_ld >= 0) { const double d = delta[P.col_ld]; step += d * d; xsq += gl[G_LD] * gl[G_LD]; gl[G_LD] += d; }
      if (P.col_ai >= 0) for (int k = 0; k < 6; ++k) { const double d = delta[P.col_ai + k]; step += d * d; xsq += gl[G_ACC_INTR + k] * gl[G_ACC_INTR + k]; gl[G_ACC_INTR + k] += d; }
      if (P.col_ci >= 0) for (int k = 0; k < P.n_intr; ++k) { const double d = delta[P.col_ci + k]; step += d * d; xsq += gl[G_CAM_INTR + k] * gl[G_CAM_INTR + k]; gl[G_CAM_INTR + k] += d; }
      if (P.col_to >= 0) { const double d = delta[P.col_to]; step += d * d; xsq += gl[G_TOFF] * gl[G_TOFF]; gl[G_TOFF] += d; }
      if (P.col_gi >= 0) for (int k = 0; k < 9; ++k) { const double d = delta[P.col_gi + k]; step += d * d; xsq += gl[G_GYR_INTR + k] * gl[G_GYR_INTR + k]; gl[G_GYR_INTR + k] += d; }
      for (int k = 0; k < G_COUNT; ++k) cand.glob[k] = gl[k];
    }
  }
  for (int o = 16; o > 0; o >>= 1) { step += __shfl_xor_sync(0xffffffffu, step, o); xsq += __shfl_xor_sync(0xffffffffu, xsq, o); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(scal + SC_STEP_SQ, step); atomicAdd(scal + SC_X_SQ, xsq); }
}

int pow2_at_least(int v) { int p = 1; while (p < v) p <<= 1; return p; }

size_t smem_A(const DeviceProblem& P, const SolvePlan& pl) { return factor_smem_bytes(pl.WS_A, P.kd + KB + pl.nbl, pl.nbl, P.kd, 0, !pl.cl_global); }
size_t smem_R(const DeviceProblem& P, const SolvePlan& pl) { return front_doubles(pl.w, 2 * pl.w + P.nb + 1) * sizeof(double) + 64; }
size_t smem_B(const DeviceProblem& P, const SolvePlan& pl) {
  const int nbp = P.nb + 1, nkr = pl.S[pl.L + 1] * pl.w;
  const size_t fac = nkr > 0 ? front_doubles(pl.w, nbp) : 0;
  const size_t back = nkr > 0 ? (size_t)nkr + 4 + (size_t)(64 + pl.kdr) * pl.ldbr + 64 : 0;   // back-substitution reuses the front area
  return ((pl.cs_global ? 0 : (size_t)nbp * nbp) + nbp + 8 + (fac > back ? fac : back)) * sizeof(double) + 64;
}
size_t smem_C(const DeviceProblem& P, const SolvePlan& pl) {
  const int maxlen = pl.len + 1 + pl.w;
  return ((size_t)pl.nbl + 4 + (size_t)pl.w + 4 + (size_t)maxlen + 4 + (size_t)(128 + P.kd) * P.ldb + 128 + (pl.stage0 ? (size_t)std::min(pl.len + 1, 128) * pl.nbl : 0)) * sizeof(double) + 64;
}
size_t smem_CR(const DeviceProblem& P, const SolvePlan& pl) {
  return ((size_t)pl.nbl + 4 + (size_t)pl.w + 4 + (size_t)2 * pl.w + 4 + (size_t)(64 + pl.kdr) * pl.ldbr + 64 + (size_t)pl.w * pl.nbl) * sizeof(double) + 64;
}

// Chunking of the knot columns: leaves cost their interior length in sequential column eliminations, every cyclic-reduction
// level a dense w = kd column front plus two launches.
// Wide borders keep chunking: the dense border blocks move to HBM (cl_global / cs_global) and the chunk count halves only
// when a kernel's shared memory still exceeds the limit.
// forced > 0 replaces the chunk count of the cost model and of ICC_SOLVER_CHUNKS / ICC_SOLVER_LEAF (tests pin every plan with it).
int env_int(const char* name, int dflt) { const char* v = getenv(name); return v && *v ? atoi(v) : dflt; }
SolvePlan make_plan(const DeviceProblem& P, int forced) {
  SolvePlan pl; memset(&pl, 0, sizeof pl);
  const int nk = P.nk, kd = P.kd, nb = P.nb;
  static const int env_chunks = env_int("ICC_SOLVER_CHUNKS", 0), leaf_cols = env_int("ICC_SOLVER_LEAF", 0);
  const int forced_chunks = forced > 0 ? forced : env_chunks;
  int Pn = 1;
  if (nk > 0 && kd > 0) {
    // P = 2^k chunks give a complete elimination tree of k-1 reduction levels; measured on B200: ~0.45 us per leaf column
    // (forward + backward) against ~25 us per level  =>  pick the k that minimises the sum while leaves keep >= kd+1 columns
    double best = 1e300;
    for (int k = 0; k <= 7; ++k) {
      const int Pc = 1 << k, len = (nk - (Pc - 1) * kd) / Pc;
      if (k > 0 && len < kd + 1) break;
      const double cost = 0.45 * len + 25.0 * std::max(0, k - 1) + (k > 0 ? 25.0 : 0.0);
      if (cost < best) { best = cost; Pn = Pc; }
    }
    if (leaf_cols > 0) Pn = (nk + kd) / (leaf_cols + kd);
    if (forced_chunks > 0) Pn = forced_chunks;
    Pn = std::max(1, std::min(Pn, 1 << (MAX_LEVELS - 1)));
    while (Pn > 1 && (nk - (Pn - 1) * kd) / Pn < kd + 1) --Pn;
  }
  auto fill = [&](int Pc) {
    memset(&pl, 0, sizeof pl);
    pl.P = Pc; pl.w = Pc > 1 ? kd : 0;
    const int interior_total = nk - (Pc - 1) * pl.w;
    pl.len = interior_total / Pc; pl.rem = interior_total % Pc;
    pl.kdr = Pc > 1 ? 2 * pl.w - 1 : 0; pl.ldbr = pl.kdr + 1;
    pl.nbl = pl.w + nb + 1;
    int l = 1, Sl = Pc - 1, off = 0;
    pl.S[1] = Sl; pl.off[1] = 0;
    while (Sl > 1) { off += Sl * pl.w; Sl /= 2; ++l; pl.S[l] = Sl; pl.off[l] = off; }
    pl.L = l - 1; pl.nkr_total = off + Sl * pl.w;
    pl.WS_A = pow2_at_least(kd + 2 * KB + 1); pl.WS_R = pl.WS_B = 0;
    pl.valid = 1;
  };
  // shared-memory fit: first choice everything on chip; wide borders move the dense border blocks to HBM (L2 resident) and drop the
  // level-0 staging; then fewer chunks; if nothing fits the opt-in limit the plan is invalid and the solve fails loudly
  const size_t COMFORT = 200 * 1024, LIMIT = 230000;
  auto fits = [&](int Pc) {
    fill(Pc);
    pl.stage0 = 1;
    if (smem_A(P, pl) > COMFORT) pl.cl_global = 1;
    if (smem_B(P, pl) > COMFORT) pl.cs_global = 1;
    if (smem_C(P, pl) > LIMIT) pl.stage0 = 0;
    pl.valid = smem_A(P, pl) <= LIMIT && smem_R(P, pl) <= LIMIT && smem_B(P, pl) <= LIMIT && smem_C(P, pl) <= LIMIT && smem_CR(P, pl) <= LIMIT;
    return pl.valid != 0;
  };
  if (!fits(Pn) && Pn > 1) { int Pc = Pn; while (Pc > 1 && !fits(Pc)) Pc /= 2; if (!pl.valid) fits(1); }
  if (!pl.valid) return pl;
  // grow the level-0 window while it fits comfortably (larger column groups amortise the group load/store)
  while (pl.WS_A < 256 && pl.WS_A < pl.len + 1 + kd + 2 * KB) { SolvePlan t = pl; t.WS_A *= 2; if (smem_A(P, t) > COMFORT) break; pl = t; }
  return pl;
}

}  // namespace

size_t solve_workspace_doubles(const DeviceProblem& P, int forced_chunks) {
  const SolvePlan pl = make_plan(P, forced_chunks);
  if (!pl.valid) return 16;
  return carve(nullptr, P.nk, P.nb, P.ldb, pl).total;
}

void solve_plan_info(const DeviceProblem& P, int forced_chunks, int32_t plan[16]) {
  const SolvePlan pl = make_plan(P, forced_chunks);
  const int32_t v[16] = {pl.valid, pl.P, pl.w, pl.len, pl.rem, pl.L, P.kd, P.nb, P.nk, pl.WS_A, pl.cl_global, pl.cs_global, pl.stage0, 0, 0, 0};
  memcpy(plan, v, sizeof v);
}

void launch_compute_scale(const DeviceProblem& P, double* scale, int jacobi, double* scal, cudaStream_t st) {
  const int n = P.nk + P.nb;
  int grid = (n + 255) / 256; if (grid > 148) grid = 148; if (grid < 1) grid = 1;
  scale_kernel<<<grid, 256, 0, st>>>(P, scale, jacobi, scal);
  count_launch();
}

int launch_solve(const DeviceProblem& P, const double* scale, SolveParams sp, double* workspace, double* delta, double* scal, cudaStream_t st, int forced_chunks) {
  const SolvePlan pl = make_plan(P, forced_chunks);
  if (!pl.valid) return 1;                       // border too wide / problem too small for any plan within the shared-memory limit
  const SolveWs ws = carve(workspace, P.nk, P.nb, P.ldb, pl);
  static size_t cfgA = 0, cfgR = 0, cfgB = 0, cfgC = 0, cfgCR = 0;
  const size_t sA = smem_A(P, pl), sR = smem_R(P, pl), sB = smem_B(P, pl), sC = smem_C(P, pl), sCR = smem_CR(P, pl);
  if (sA > cfgA) { cudaFuncSetAttribute(eliminate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sA); cfgA = sA; }
  if (sR > cfgR) { cudaFuncSetAttribute(reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sR); cfgR = sR; }
  if (sB > cfgB) { cudaFuncSetAttribute(root_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sB); cfgB = sB; }
  if (sC > cfgC) { cudaFuncSetAttribute(backsub_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sC); cfgC = sC; }
  if (sCR > cfgCR) { cudaFuncSetAttribute(backsub_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sCR); cfgCR = sCR; }
  cudaMemsetAsync(ws.bandr, 0, ws.reduced_doubles * sizeof(double), st);
  if (P.nk == 0) cudaMemsetAsync(scal, 0, 5 * sizeof(double), st);   // otherwise the first solver kernel clears the step scalars
  if (P.nk > 0) {
    launch_pdl(prepare_kernel, dim3(pl.P, pl.P >= 64 ? 4 : 16), 256, 0, st, P, pl, scale, sp, workspace, scal); count_launch();
    launch_pdl(eliminate_kernel, pl.P, NT, sA, st, P, pl, workspace, scal); count_launch();
    for (int l = 1; l <= pl.L; ++l) { launch_pdl(reduce_kernel, (pl.S[l] + 1) / 2, NT, sR, st, P, pl, l, workspace, scal); count_launch(); }
  }
  launch_pdl(root_kernel, 1, NT, sB, st, P, pl, scale, sp, workspace, scal); count_launch();
  if (P.nk > 0) {
    for (int l = pl.L; l >= 1; --l) { launch_pdl(backsub_kernel<false>, (pl.S[l] + 1) / 2, NT, sCR, st, P, pl, l, workspace, (const double*)scal); count_launch(); }
    launch_pdl(backsub_kernel<true>, pl.P, NT, sC, st, P, pl, 0, workspace, (const double*)scal); count_launch();
  }
  const int n = P.nk + P.nb;
  int grid = (n + 255) / 256; if (grid > 148) grid = 148; if (grid < 1) grid = 1;
  launch_pdl(finish_kernel, grid, 256, 0, st, P, pl, scale, sp, workspace, delta, scal); count_launch();
  return cudaGetLastError() == cudaSuccess ? 0 : 2;
}

void launch_update(const DeviceProblem& P, const DeviceState& cur, const DeviceState& cand, const double* delta, double max_ba, double max_bg, double* scal, cudaStream_t st) {
  const int total = P.n_so3 + P.n_r3 + P.n_ba + P.n_bg + 1;
  launch_pdl(update_kernel, (total + 127) / 128, 128, 0, st, P, cur, cand, delta, max_ba, max_bg, scal);
  count_launch();
}

}  // namespace icc
