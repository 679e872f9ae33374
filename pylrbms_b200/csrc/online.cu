// Online half of the LRBMS hot path: mu-batched assembly + sparse Cholesky + solves of the block-sparse reduced
// system (K3 + K4), mu-batched estimator quadratic forms (K5) and the eta combine / max reduction.
//
// solve_kernel_v2: one CTA per parameter (grid-stride over the batch).  The reduced matrix lives as 8x8 tiles (the
// DMMA.8x8x4 accumulator shape); the host-side symbolic phase (symbolic.cpp) provides, per tile column, its targets and
// their (L_IK, L_JK) update pairs as slots of a shared-memory window of live factor tiles.  Every target
// A_IJ(mu) - sum_K L_IK L_JK^T is accumulated with DMMA (A_IJ(mu) = sum_q theta_q(mu) A_q is assembled on the fly, left
// to right like LincombOperator.assemble), the diagonal tile is factored and inverted, and the off-diagonal tiles are
// multiplied by L_JJ^{-T}.  The right-hand side rides along as one more tile row (forward substitution fused into the
// factorisation).  Systems whose window does not fit one SM's shared memory go to the band solver (band.cu).  The kernel
// factors P A P^T with the subdomains in the elimination order the symbolic phase chose (lrbms_symbolic_choose_order);
// the operator tiles and the rhs are uploaded permuted, u and the failed-pivot row go back through a row map.
//
// estimate_kernel: one CTA per (subdomain, tile of 32 parameters).  Every quadratic form x_L^T M x_R of
// reference estimators.py:71-85 is evaluated for 32 parameters at once as Y = M X_R on DMMA followed by a column dot
// with X_L; the matrices are read once per 32 parameters instead of once per parameter.
#include <algorithm>
#include <cmath>

#include "band.h"
#include "common.cuh"
#include "symbolic.h"

namespace {

// ------------------------------------------------------------------------------------------------------
//  solve_kernel_v2: left-looking 8x8-tile Cholesky around shared memory.
//    * one CTA of 16 warps per SM; the *live window* of L -- off-diagonal tiles (I, K) with K < J <= I, 253 tiles
//      for the C2 band -- stays in shared memory in DMMA operand-fragment order (one conflict-free LDS.128 per lane
//      and operand); the factor goes to global memory only once, for the backward substitution;
//    * software pipeline over tile columns: while warp 0 factors and inverts the diagonal tile of column J-1, all
//      other warps already accumulate the "early" updates of column J (source columns <= J-2); the "late" update
//      with column J-1 (one pair per target) follows the triangular solve of column J-1;
//    * targets of a column are handed out dynamically (longest first) through a shared-memory counter;
//    * the backward substitution streams the factor back with a 4-stage cp.async ring.
// ------------------------------------------------------------------------------------------------------
// (kV2Warps, kBackStages, kMetaBufs and kABufs are in symbolic.h: the symbolic phase sizes the shared memory with them)
constexpr int kV2Threads = kV2Warps * 32;

struct SolveParamsV2 {
  int32_t n_red, n_pad, Q, Qf, n_theta, n_a_tiles, ntc;
  const int32_t* row_idx;   // [n_tiles] tile row of every factor slot
  const int32_t* row_map;   // [n_red] row of u (the caller's order) of every row of the permuted system
  const double* a_tiles;    // [Q][n_a_tiles][64]
  const double* rhs;        // [Qf][n_pad]
  int64_t work_stride;      // doubles of factor scratch per CTA: n_tiles * 64
  const int4* ccol;         // [ntc + 1] {first tile, tiles, first item, tile (J+1, J) exists}
  const int4* ccol2;        // [ntc] {first tile pair, tile pairs, first rhs pair, rhs pairs}
  const int4* ccol3;        // [ntc] {first staged operator tile, staged operator tiles, 0, 0}
  const int32_t* ca_tile;   // operator tile index (into a_tiles) per staged tile
  int32_t n_ca;             // length of ca_tile
  const int4* cdesc;        // per item: {pair begin, late begin, pair end (staged offsets), staged operator tile or -1}
  const int32_t* cslot;     // per item: (window slot + 1; 0: diagonal tile / rhs row) | (has a source-(J-2) pair) << 20
  const int32_t* cord;      // per item position: li in hand-out order (longest early update first)
  const int32_t* cnext;     // per item: li of the target in the next column its tile feeds (-1: none)
  const int2* win_ab;       // per pair: window slots of the two operands (a < 0: forward-solve row y_{-a-1})
  int32_t region_doubles;   // shared-memory window region (also the backward-substitution ring)
  int32_t max_targets;      // per column, incl. the diagonal tile and the rhs row
  int32_t max_col_pairs;
  int32_t a_ring;           // operator-tile slots of the staging ring (lrbms_symbolic::a_ring)
  int32_t back_stage_doubles;
  int32_t staggered;        // schedule variant of the symbolic phase (lrbms_symbolic::staggered)
#ifdef LRBMS_DEVTOOLS
  long long* timing;        // developer builds only (-DLRBMS_DEVTOOLS, LRBMS_SOLVE_TIMING=1): [16 warps][8 phases] SM cycles of CTA 0
#endif
};

// acc -= sum_p A_p * B_p^T over staged pairs [p0, p1).  Eight accumulator registers = four independent DMMA chains
// (two pairs in flight x two k halves): the dependent-issue latency of DMMA, not its throughput, is what a single
// warp runs into.  RHS = true: the A operand is the forward-solve row y_K (row 0 of a virtual tile).
template <bool RHS>
__device__ __forceinline__ void apply_pairs(const int2* __restrict__ pairs, const double* __restrict__ win,
                                            const double* __restrict__ sx, int p0, int p1, int lane, double (&acc)[8]) {
  const int g = lane >> 2, t = lane & 3;
  auto load_a = [&](int a) -> double2 {
    if (!RHS) return *reinterpret_cast<const double2*>(win + a * 64 + lane * 2);
    const int K = -a - 1;
    return make_double2((g == 0) ? sx[8 * K + t] : 0.0, (g == 0) ? sx[8 * K + 4 + t] : 0.0);
  };
  int p = p0;
#pragma unroll 2
  for (; p + 1 < p1; p += 2) {
    const int2 ab0 = pairs[p], ab1 = pairs[p + 1];
    const double2 fa = load_a(ab0.x), ga = load_a(ab1.x);
    const double2 fb = *reinterpret_cast<const double2*>(win + ab0.y * 64 + lane * 2);
    const double2 gb = *reinterpret_cast<const double2*>(win + ab1.y * 64 + lane * 2);
    dmma884(acc[0], acc[1], -fa.x, fb.x);
    dmma884(acc[4], acc[5], -ga.x, gb.x);
    dmma884(acc[2], acc[3], -fa.y, fb.y);
    dmma884(acc[6], acc[7], -ga.y, gb.y);
  }
  if (p < p1) {
    const int2 ab0 = pairs[p];
    const double2 fa = load_a(ab0.x);
    const double2 fb = *reinterpret_cast<const double2*>(win + ab0.y * 64 + lane * 2);
    dmma884(acc[0], acc[1], -fa.x, fb.x);
    dmma884(acc[2], acc[3], -fa.y, fb.y);
  }
}

__global__ void __launch_bounds__(kV2Threads, 1)
solve_kernel_v2(SolveParamsV2 P, int64_t n_mu, const double* __restrict__ theta, double* __restrict__ u,
                int32_t* __restrict__ info, double* __restrict__ work) {
  extern __shared__ __align__(16) double smem[];
  const int MT = P.max_targets;
  double* win = smem;                                         // region_doubles
  double* acc0 = win + P.region_doubles;                      // 3 * MT * 64: target sums of columns J-1, J, J+1
  double* sx = acc0 + 3 * MT * 64;                            // n_pad
  double* sW = sx + P.n_pad;                                  // 2 * 64: L_JJ^{-1} of the current and the previous column
  double* sScr = sW + 2 * 64;                                 // 2 * 64: layout-conversion scratch (shared tile, chain warp)
  double* sred = sScr + 2 * 64;                               // 2 * kV2Warps * 8
  double* sth = sred + 2 * kV2Warps * 8;                      // n_theta (<= 32)
  double* sA = sth + 32;                                      // a_ring * Q * 64
  const int a_tile_doubles = P.Q * 64;
  int4* sDesc = reinterpret_cast<int4*>(sA + P.a_ring * a_tile_doubles);          // kMetaBufs * MT
  int4* sCol = sDesc + kMetaBufs * MT;                                            // ntc + 1
  int4* sCol2 = sCol + (P.ntc + 1);                                               // ntc
  int4* sCol3 = sCol2 + P.ntc;                                                    // ntc
  int2* sPair = reinterpret_cast<int2*>(sCol3 + P.ntc);                           // kMetaBufs * max_col_pairs
  int* sSlot = reinterpret_cast<int*>(sPair + kMetaBufs * P.max_col_pairs);       // kMetaBufs * MT
  int* sOrd = sSlot + kMetaBufs * MT;                                             // kMetaBufs * MT
  int* sNext = sOrd + kMetaBufs * MT;                                             // kMetaBufs * MT
  int* sCaTile = sNext + kMetaBufs * MT;                                          // n_ca
  __shared__ int s_info;
  __shared__ __align__(8) unsigned long long s_back_bar[kBackStages];            // mbarriers of the backward-substitution ring

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  double* L = work + (int64_t)blockIdx.x * P.work_stride;
#ifdef LRBMS_DEVTOOLS
  const bool timing = P.timing != nullptr && blockIdx.x == 0;
  long long tph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = 0;
// (bar.sync compiles to BAR.SYNC.DEFER_BLOCKING: a clock read right behind it is taken before the wait; the volatile
// shared-memory read makes the barrier complete first)
#define LRBMS_TICK(k) do { if (timing) { const int dummy_ = *(volatile int*)&s_info; const long long now_ = clock64() + (dummy_ & 0); tph[k] += now_ - tlast; tlast = now_; } } while (0)
#else
#define LRBMS_TICK(k) do { } while (0)
#endif

  // ---- per-column tables: loaded once per CTA, no global-memory latency inside the column loop afterwards
  for (int i = threadIdx.x; i <= P.ntc; i += kV2Threads) sCol[i] = P.ccol[i];
  for (int i = threadIdx.x; i < P.ntc; i += kV2Threads) { sCol2[i] = P.ccol2[i]; sCol3[i] = P.ccol3[i]; }
  for (int i = threadIdx.x; i < P.n_ca; i += kV2Threads) sCaTile[i] = P.ca_tile[i];
  __syncthreads();

  // stage everything column Jn needs into buffer Jn % kMetaBufs and the operator-tile ring.  Called by ONE producer warp (the
  // address arithmetic is a long dependent chain; keeping it off the other 15 warps takes it off the critical path);
  // asynchronous copies, one commit group per call
  auto stage_meta = [&](int Jn) {
    if (Jn < P.ntc) {
      const int b = Jn % kMetaBufs;
      const int4 col = sCol[Jn];
      const int4 ci = sCol2[Jn];
      const int4 c3 = sCol3[Jn];
      for (int i = lane; i <= col.y; i += 32) {
        cp_async16(sDesc + b * MT + i, P.cdesc + col.z + i);
        cp_async4(sSlot + b * MT + i, P.cslot + col.z + i);
        cp_async4(sOrd + b * MT + i, P.cord + col.z + i);
        cp_async4(sNext + b * MT + i, P.cnext + col.z + i);
      }
      int2* dst = sPair + b * P.max_col_pairs;
      for (int i = lane; i < ci.y; i += 32) cp_async8(dst + i, P.win_ab + ci.x + i);
      for (int i = lane; i < ci.w; i += 32) cp_async8(dst + ci.y + i, P.win_ab + ci.z + i);
      // raw operator tiles A_q of the column's targets (the theta-weighted sum is formed when they are consumed):
      // one 16-byte chunk per lane, 32 lanes = one tile per step.  Tile k of the column goes to ring slot
      // (c3.x + k) mod a_ring: the tiles of the kABufs columns alive at a time never share a slot.
      int slot = c3.x % P.a_ring;
      for (int k = 0; k < c3.y; ++k) {
        const int64_t src_tile = sCaTile[c3.x + k];
        for (int q = 0; q < P.Q; ++q)
          cp_async16(sA + (slot * P.Q + q) * 64 + lane * 2, P.a_tiles + ((int64_t)q * P.n_a_tiles + src_tile) * 64 + lane * 2);
        if (++slot == P.a_ring) slot = 0;
      }
    }
    cp_async_commit();
  };
  constexpr int kProducer = kV2Warps - 1;   // warp 15 only stages data; warp 0 only runs the critical chain
  constexpr int kUpd = kV2Warps - 2;        // update warps 1..14
  const bool is_upd = warp > 0 && warp < kProducer;

  // ---- building blocks of the column pipeline -----------------------------------------------------------------
  // early updates of column Jx (source columns <= Jx - 2) by the 15 update warps -> accX
  auto early_updates = [&](int Jx, double* accX) {
    const int mb = Jx % kMetaBufs;
    const int4* descC = sDesc + mb * MT;
    const int2* pairC = sPair + mb * P.max_col_pairs;
    const int* ordC = sOrd + mb * MT;
    const int a_first = sCol3[Jx].x % P.a_ring;               // ring slot of the column's first staged operator tile
    const int ncol = sCol[Jx].y;
    // Snake deal over the 14 update warps (1..14), longest item first.  (The triangular solve gives warps
    // 1 .. n_tiles - 14 two tiles and the others one, so the longest early items go to the *high* warps: warp 14 first.)
    const int posU = kUpd - warp;
    const int posR = kUpd - 1 - posU;
    for (int r = 0; kUpd * r <= ncol; ++r) {
      const int item = kUpd * r + ((r & 1) ? posR : posU);
      if (item > ncol) continue;
      const int li = ordC[item];
      const int4 d = descC[li];
      double2 v0 = make_double2(0.0, 0.0), v1 = v0;           // rhs row: loads issued first, consumed last
      if (li == ncol && g == 0) {
        v0 = __ldg(reinterpret_cast<const double2*>(P.rhs + 8 * Jx + 2 * t));
        if (P.Qf > 1) v1 = __ldg(reinterpret_cast<const double2*>(P.rhs + P.n_pad + 8 * Jx + 2 * t));
      }
      double acc[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] = 0.0;
      if (li < ncol) apply_pairs<false>(pairC, win, sx, d.x, d.y, lane, acc);
      else apply_pairs<true>(pairC, win, sx, d.x, d.y, lane, acc);
      double a0 = 0.0, a1 = 0.0;
      if (li < ncol) {
        if (d.w >= 0) {                                        // A(mu) tile = sum_q theta_q A_q, left to right
          const int slot = (a_first + d.w < P.a_ring) ? a_first + d.w : a_first + d.w - P.a_ring;
          const double* at = sA + slot * a_tile_doubles + g * 8 + 2 * t;
          for (int q = 0; q < P.Q; ++q) {
            const double2 v = *reinterpret_cast<const double2*>(at + q * 64);
            if (q == 0) { a0 = sth[0] * v.x; a1 = sth[0] * v.y; }
            else { a0 += sth[q] * v.x; a1 += sth[q] * v.y; }
          }
        }
      } else {
        a0 = sth[P.Q] * v0.x; a1 = sth[P.Q] * v0.y;
        if (P.Qf > 1) { a0 += sth[P.Q + 1] * v1.x; a1 += sth[P.Q + 1] * v1.y; }
        for (int q = 2; q < P.Qf && g == 0; ++q) {
          const double2 v = __ldg(reinterpret_cast<const double2*>(P.rhs + (int64_t)q * P.n_pad + 8 * Jx + 2 * t));
          a0 += sth[P.Q + q] * v.x; a1 += sth[P.Q + q] * v.y;
        }
      }
      *reinterpret_cast<double2*>(accX + li * 64 + lane * 2) =
          make_double2(a0 + ((acc[0] + acc[4]) + (acc[2] + acc[6])), a1 + ((acc[1] + acc[5]) + (acc[3] + acc[7])));
    }
  };

  // column Jy: triangular solve L_IJ = C_IJ L_JJ^{-T} of its off-diagonal tiles and its rhs row (update warps), fused
  // with the "late" update of column Jy + 1: target (I, Jy+1) -= L_{I,Jy} L_{Jy+1,Jy}^T, done by the warp that just formed
  // L_{I,Jy}.  The late update of the *diagonal* target belongs to warp 0's critical chain and is skipped here.
  auto solve_column = [&](int Jy, const double* accY, double* accL, const double* sWy) {
    const int4 col = sCol[Jy];
    const int cp0 = col.x, ncol = col.y;
    const int has_next = (Jy + 1 < P.ntc) ? col.w : 0;
    const int mbp = Jy % kMetaBufs;
    const int* slotP = sSlot + mbp * MT;
    const int* nextP = sNext + mbp * MT;
    // metadata of column Jy + 1: its targets get, besides the late update with the tile formed here, their pair with
    // source column Jy - 1 (both operands in the window) -- the early updates stop one source column earlier
    const int mbn = (Jy + 1) % kMetaBufs;
    const int* slotN = sSlot + mbn * MT;
    const int4* descN = sDesc + mbn * MT;
    const int2* pairN = sPair + mbn * P.max_col_pairs;
    const int ncolN = (Jy + 1 < P.ntc) ? sCol[Jy + 1].y : 0;
    double2 fbn = make_double2(0.0, 0.0);
    // Slot 0: L_{Jy+1,Jy} (every warp forms it itself instead of waiting for another warp); slots 1, 2: two of this
    // warp's own items.  The three solves are independent, written side by side so their latencies overlap.
    for (int base = warp; base <= ncol; base += 2 * kUpd) {
      const int li[3] = {1, base, base + kUpd};
      const bool on[3] = {has_next != 0 && base == warp, true, base + kUpd <= ncol};
      // X = C W^T.  C is read from its row-major accumulator tile directly in DMMA A-fragment order and X goes back
      // through shared memory to reach the operand-fragment order -- no shuffles (they queue behind the LDS traffic).
      double x0[3] = {0.0, 0.0, 0.0}, x1[3] = {0.0, 0.0, 0.0};
      double a0[3], a1[3];
      double2 cc[3];
      int nl[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const double* ct = accY + li[k] * 64 + g * 8 + t;
        a0[k] = on[k] ? ct[0] : 0.0;
        a1[k] = on[k] ? ct[4] : 0.0;
        nl[k] = (k > 0 && on[k] && has_next) ? nextP[li[k]] : -1;
        if (nl[k] == 0) nl[k] = -1;                            // diagonal target: warp 0 does it
        cc[k] = (nl[k] > 0) ? *reinterpret_cast<const double2*>(accL + nl[k] * 64 + lane * 2) : make_double2(0.0, 0.0);
      }
      const double b0 = sWy[g * 8 + t], b1 = sWy[g * 8 + 4 + t];
#pragma unroll
      for (int k = 0; k < 3; ++k) dmma884(x0[k], x1[k], a0[k], b0);
#pragma unroll
      for (int k = 0; k < 3; ++k) dmma884(x0[k], x1[k], a1[k], b1);
      __syncwarp();                                            // all lanes have read their C fragments
      double* tile[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        // own tiles are dead after this solve and serve as scratch; the shared tile (1) is read by every warp, so its
        // result goes to a common scratch tile (all warps write identical values)
        tile[k] = (li[k] == 1) ? sScr : const_cast<double*>(accY) + li[k] * 64;
        if (on[k]) *reinterpret_cast<double2*>(tile[k] + lane * 2) = make_double2(x0[k], x1[k]);
      }
      __syncwarp();
      double2 frag[3];
#pragma unroll
      for (int k = 0; k < 3; ++k)
        frag[k] = on[k] ? make_double2(tile[k][g * 8 + t], tile[k][g * 8 + t + 4]) : make_double2(0.0, 0.0);
      if (base == warp) fbn = frag[0];
#pragma unroll
      for (int k = 1; k < 3; ++k) {
        if (!on[k]) continue;
        if (li[k] < ncol) {
          *reinterpret_cast<double2*>(win + ((slotP[li[k]] & 0xfffff) - 1) * 64 + lane * 2) = frag[k];
          *reinterpret_cast<double2*>(L + (int64_t)(cp0 + li[k]) * 64 + lane * 2) = frag[k];
        } else if (g == 0) {
          sx[8 * Jy + 2 * t] = x0[k];
          sx[8 * Jy + 2 * t + 1] = x1[k];
        }
        if (nl[k] > 0) {
          double n0 = 0.0, n1 = 0.0;
          dmma884(cc[k].x, cc[k].y, -frag[k].x, fbn.x);
          dmma884(n0, n1, -frag[k].y, fbn.y);
          if (slotN[nl[k]] >> 20) {                       // pair with source column Jy - 1, from the window
            const int2 ab = pairN[descN[nl[k]].y];
            double2 fa;
            if (nl[k] < ncolN) fa = *reinterpret_cast<const double2*>(win + ab.x * 64 + lane * 2);
            else {                                        // rhs row: the A operand is the forward-solve row y_K
              const int K = -ab.x - 1;
              fa = make_double2((g == 0) ? sx[8 * K + t] : 0.0, (g == 0) ? sx[8 * K + 4 + t] : 0.0);
            }
            const double2 fb = *reinterpret_cast<const double2*>(win + ab.y * 64 + lane * 2);
            dmma884(cc[k].x, cc[k].y, -fa.x, fb.x);
            dmma884(n0, n1, -fa.y, fb.y);
          }
          *reinterpret_cast<double2*>(accL + nl[k] * 64 + lane * 2) = make_double2(cc[k].x + n0, cc[k].y + n1);
        }
      }
    }
  };

  // warp 0's critical chain for column Jc: finish the diagonal target (late update with L_{Jc,Jc-1}), then factor it by
  // row operations on [A | I] held one row per lane, so L^{-1} falls out of the same eight steps -> sWc, and the diagonal
  // slot of the stored factor
  auto diagonal_chain = [&](int Jc, const double* accPrev, double* accCur, const double* sWp, double* sWc) {
    if (Jc >= 1 && sCol[Jc - 1].w) {
      const double* ct = accPrev + 64 + g * 8 + t;                                       // target (Jc, Jc-1)
      double x0 = 0.0, x1 = 0.0;
      dmma884(x0, x1, ct[0], sWp[g * 8 + t]);
      dmma884(x0, x1, ct[4], sWp[g * 8 + 4 + t]);
      double* scr = sScr + 64;
      *reinterpret_cast<double2*>(scr + lane * 2) = make_double2(x0, x1);
      __syncwarp();
      const double2 frag = make_double2(scr[g * 8 + t], scr[g * 8 + t + 4]);
      double2 cc = *reinterpret_cast<const double2*>(accCur + lane * 2);
      double n0 = 0.0, n1 = 0.0;
      dmma884(cc.x, cc.y, -frag.x, frag.x);
      dmma884(n0, n1, -frag.y, frag.y);
      *reinterpret_cast<double2*>(accCur + lane * 2) = make_double2(cc.x + n0, cc.y + n1);
      __syncwarp();
    }
    if (sSlot[(Jc % kMetaBufs) * MT] >> 20) {                                              // pair with source column Jc - 2
      const int2 ab = sPair[(Jc % kMetaBufs) * P.max_col_pairs + sDesc[(Jc % kMetaBufs) * MT].y];
      const double2 fa = *reinterpret_cast<const double2*>(win + ab.x * 64 + lane * 2);
      const double2 fb = *reinterpret_cast<const double2*>(win + ab.y * 64 + lane * 2);
      double2 cc = *reinterpret_cast<const double2*>(accCur + lane * 2);
      double n0 = 0.0, n1 = 0.0;
      dmma884(cc.x, cc.y, -fa.x, fb.x);
      dmma884(n0, n1, -fa.y, fb.y);
      __syncwarp();
      *reinterpret_cast<double2*>(accCur + lane * 2) = make_double2(cc.x + n0, cc.y + n1);
      __syncwarp();
    }
    // Scalar Cholesky of the 8x8 tile, done redundantly by every lane in registers (packed lower triangle): no
    // cross-lane traffic on this chain -- shuffles would queue behind the shared-memory traffic of the update warps.
    double l[36], rinv[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j <= i; ++j) l[i * (i + 1) / 2 + j] = accCur[i * 8 + j];
    int bad = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      double akk = l[k * (k + 1) / 2 + k];
      if (8 * Jc + k >= P.n_red) akk = 1.0;                  // padding rows: identity
      if (!(akk > 0.0)) { if (!bad) bad = 8 * Jc + k + 1; akk = 1.0; }
      const double r = rsqrt(akk);
      rinv[k] = r;
#pragma unroll
      for (int i = k + 1; i < 8; ++i) l[i * (i + 1) / 2 + k] *= r;
#pragma unroll
      for (int j = k + 1; j < 8; ++j)
#pragma unroll
        for (int i = j; i < 8; ++i) l[i * (i + 1) / 2 + j] -= l[i * (i + 1) / 2 + k] * l[j * (j + 1) / 2 + k];
    }
    if (bad && lane == 0 && s_info == 0) s_info = bad;
    // column c = lane & 7 of W = L^{-1} by forward substitution (entries above the diagonal come out as exact zeros)
    const int c = lane & 7;
    double w[8];
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
      double sacc = (ii == c) ? 1.0 : 0.0;
#pragma unroll
      for (int k = 0; k < ii; ++k) sacc -= l[ii * (ii + 1) / 2 + k] * w[k];
      w[ii] = sacc * rinv[ii];
    }
    if (lane < 8) {
      const int64_t dslot = (int64_t)sCol[Jc].x * 64;
#pragma unroll
      for (int ii = 0; ii < 8; ++ii) {
        sWc[ii * 8 + c] = w[ii];
        L[dslot + ii * 8 + c] = w[ii];                        // the diagonal slot of the stored factor holds L_JJ^{-1}
      }
    }
  };

  for (int64_t mu = blockIdx.x; mu < n_mu; mu += gridDim.x) {
    __syncthreads();
    for (int q = threadIdx.x; q < P.n_theta; q += kV2Threads) sth[q] = theta[mu * P.n_theta + q];
    if (threadIdx.x == 0) s_info = 0;
    if (warp == kProducer) { stage_meta(0); stage_meta(1); stage_meta(2); }
    cp_async_wait<0>();
    __syncthreads();
#ifdef LRBMS_DEVTOOLS
    if (timing) tlast = clock64();
#endif
    if (is_upd) early_updates(0, acc0);
    __syncthreads();

    // Column pipeline.  Iteration J:  warp 0 runs the critical chain of column J (late update of the diagonal target,
    // factorisation, inverse) while the update warps solve column J-1 against L_{J-1,J-1}^{-1}, apply the late updates of
    // column J, synchronise among themselves and accumulate the early updates of column J+1.
    for (int J = 0; J < P.ntc; ++J) {
      if (warp == kProducer) stage_meta(J + 3);
      LRBMS_TICK(0);
      double* accPrev = acc0 + ((J + 2) % 3) * MT * 64;       // target sums of column J-1 (pointer arithmetic on purpose:
      double* accCur = acc0 + (J % 3) * MT * 64;              // an indexed pointer array would live in local memory)
      double* accNext = acc0 + ((J + 1) % 3) * MT * 64;
      double* sWprev = sW + ((J + 1) & 1) * 64;
      double* sWcur = sW + (J & 1) * 64;
      if (warp == 0) {
        diagonal_chain(J, accPrev, accCur, sWprev, sWcur);
        LRBMS_TICK(1);
      } else if (is_upd) {
        if (P.staggered) {
          // The early updates of column J+1 (source columns <= J-2) do not touch anything the triangular solve of column
          // J-1 produces, so the two run in either order: odd update warps solve first, even ones second -- the
          // bandwidth-bound pair loops of one half overlap the latency-bound solves of the other.
          if (warp & 1) {
            if (J >= 1) solve_column(J - 1, accPrev, accCur, sWprev);
            LRBMS_TICK(1);
            if (J + 1 < P.ntc) early_updates(J + 1, accNext);
            LRBMS_TICK(3);
          } else {
            if (J + 1 < P.ntc) early_updates(J + 1, accNext);
            LRBMS_TICK(3);
            if (J >= 1) solve_column(J - 1, accPrev, accCur, sWprev);
            LRBMS_TICK(1);
          }
        } else {
          // patterns without carrier tiles: early updates include source column J-1, i.e. they follow the solve
          if (J >= 1) solve_column(J - 1, accPrev, accCur, sWprev);
          LRBMS_TICK(1);
          asm volatile("bar.sync 1, %0;\n" ::"n"(kUpd * 32) : "memory");   // column J-1 of L visible to the update warps
          LRBMS_TICK(2);
          if (J + 1 < P.ntc) early_updates(J + 1, accNext);
          LRBMS_TICK(3);
        }
      }
      cp_async_wait<1>();   // everything staged for column J+2 has landed (column J+3 may still be in flight)
      __syncthreads();
      LRBMS_TICK(4);
    }
    if (is_upd) solve_column(P.ntc - 1, acc0 + ((P.ntc - 1) % 3) * MT * 64, acc0 + (P.ntc % 3) * MT * 64, sW + ((P.ntc - 1) & 1) * 64);
    LRBMS_TICK(5);
    cp_async_wait<0>();

    // ---------------- backward substitution  L^T u = y.  The factor streams back through a cp.async ring.  Per tile
    //                  column J (descending): warp 0 finishes u_J -- partial sums of column J (formed one iteration
    //                  earlier by the other warps), the one contribution that needs u_{J+1}, then L_JJ^{-T} -- while
    //                  warps 1..15 already form the partial sums of column J-1 from u_I, I >= J+1.  One barrier per column.
    {
      const int stage = P.back_stage_doubles;
      auto issue = [&](int Jc) {
        if (Jc >= 0) {
          const int4 col = sCol[Jc];
          double* dst = win + ((P.ntc - 1 - Jc) % kBackStages) * stage;
          const double* src = L + (int64_t)col.x * 64;
          // one bulk copy (TMA engine) per tile column, completing on the stage's mbarrier; the n-th use of a stage waits
          // for parity n & 1.  (768 cp.async per column kept fifteen warps ~450 cycles per column in the copy queue.)
          const int sidx = (P.ntc - 1 - Jc) % kBackStages;
          if (threadIdx.x == 32) {
            mbar_expect_tx(&s_back_bar[sidx], (unsigned)(col.y * 512));
            bulk_copy_g2s(dst, src, (unsigned)(col.y * 512), &s_back_bar[sidx]);
          }
          const int tid = (int)threadIdx.x - 64;
          int* rdst = sSlot + sidx * MT;                               // sSlot/sOrd/sNext are free now: 15 MT ints
          if (tid >= 0 && tid < col.y) cp_async4(rdst + tid, P.row_idx + col.x + tid);
        }
        cp_async_commit();
      };
      auto wait_column = [&](int Jc) {
        if (Jc >= 0) mbar_wait(&s_back_bar[(P.ntc - 1 - Jc) % kBackStages], (unsigned)(((P.ntc - 1 - Jc) / kBackStages) & 1));
      };
      // The factor tiles written with st.global above are read back by bulk copies (async proxy): every writer orders its
      // generic-proxy stores before later async-proxy accesses (all state spaces) ahead of the barrier.
      fence_proxy_async_all();
      __syncthreads();                                  // everybody is through with the window
      if (threadIdx.x == 0)
        for (int i = 0; i < kBackStages; ++i) mbar_init(&s_back_bar[i], 1);
      fence_proxy_async();                              // ... which the bulk copies overwrite
      for (int i = threadIdx.x; i < 2 * kV2Warps * 8; i += kV2Threads) sred[i] = 0.0;
      __syncthreads();
      for (int s = 0; s < kBackStages - 2; ++s) issue(P.ntc - 1 - s);
      cp_async_wait<kBackStages - 4>();       // columns ntc-1 and ntc-2 have landed
      __syncthreads();
      for (int J = P.ntc - 1; J >= 0; --J) {
        issue(J - (kBackStages - 2));
        if (warp == 0) {
          wait_column(J);
          const int bsel = (P.ntc - 1 - J) % kBackStages;
          const double* buf = win + bsel * stage;
          const double* red = sred + (J & 1) * kV2Warps * 8;
          const int cidx = lane & 7, q4 = lane >> 3;
          // lane (q, c): four of the sixteen partials of component c, then a two-step butterfly
          const double* rq = red + (q4 * 4) * 8 + cidx;
          double part = (rq[0] + rq[8]) + (rq[16] + rq[24]);
          part += __shfl_xor_sync(0xffffffffu, part, 8);
          part += __shfl_xor_sync(0xffffffffu, part, 16);
          if (sCol[J].w) {                     // tile (J+1, J): the only contribution that needs u_{J+1}
            const double2 f = *reinterpret_cast<const double2*>(buf + 64 + lane * 2);
            const double xv = sx[8 * (J + 1) + g];
            double s0 = f.x * xv, s1 = f.y * xv;     // components t and t + 4, to be summed over g
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
              s0 += __shfl_xor_sync(0xffffffffu, s0, o);
              s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            }
            const double v0 = __shfl_sync(0xffffffffu, s0, cidx & 3), v1 = __shfl_sync(0xffffffffu, s1, cidx & 3);
            part += (cidx < 4) ? v0 : v1;
          }
          const double v = sx[8 * J + cidx] - part;            // lanes c, c + 8, c + 16, c + 24 all hold v_c
          // u_c = sum_k W[k][c] v_k: lane (q, c) takes k = 2q, 2q + 1
          double accv = buf[(2 * q4) * 8 + cidx] * __shfl_sync(0xffffffffu, v, 2 * q4) +
                        buf[(2 * q4 + 1) * 8 + cidx] * __shfl_sync(0xffffffffu, v, 2 * q4 + 1);
          accv += __shfl_xor_sync(0xffffffffu, accv, 8);
          accv += __shfl_xor_sync(0xffffffffu, accv, 16);
          if (lane < 8) sx[8 * J + cidx] = accv;
        } else {
          double s0 = 0.0, s1 = 0.0;           // partial sums of column J-1 for solution components t and t + 4
          if (J >= 1) {
            wait_column(J - 1);
            const int bsel = (P.ntc - J) % kBackStages;
            const double* buf = win + bsel * stage;
            const int* rows = sSlot + bsel * MT;
            const int4 col = sCol[J - 1];
            for (int li = 1 + col.w + (warp - 1); li < col.y; li += kV2Warps - 1) {    // skip tile (J, J-1)
              const double2 f = *reinterpret_cast<const double2*>(buf + li * 64 + lane * 2);
              const double xv = sx[8 * rows[li] + g];
              s0 += f.x * xv;
              s1 += f.y * xv;
            }
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
              s0 += __shfl_xor_sync(0xffffffffu, s0, o);
              s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            }
          }
          double* red = sred + ((J + 1) & 1) * kV2Warps * 8;   // = ((J - 1) & 1): partials of column J-1
          if (g == 0) { red[warp * 8 + t] = s0; red[warp * 8 + 4 + t] = s1; }
        }
        cp_async_wait<kBackStages - 4>();     // columns J-1 and J-2 have landed
        __syncthreads();
      }
      cp_async_wait<0>();
    }
    LRBMS_TICK(6);
    // back to the caller's row order; a failed pivot is reported as its row there
    for (int i = threadIdx.x; i < P.n_red; i += kV2Threads) u[mu * P.n_red + __ldg(P.row_map + i)] = sx[i];
    if (threadIdx.x == 0 && info) info[mu] = s_info ? __ldg(P.row_map + s_info - 1) + 1 : 0;
    LRBMS_TICK(7);
  }
#ifdef LRBMS_DEVTOOLS
  if (timing && lane == 0)
    for (int k = 0; k < 8; ++k) P.timing[warp * 8 + k] = tph[k];
#endif
#undef LRBMS_TICK
}

// ------------------------------------------------------------------------------------------------------
//  estimator
// ------------------------------------------------------------------------------------------------------
constexpr int kEstThreads = 512;
constexpr int kEstWarps = kEstThreads / 32;
// parameters per CTA (template argument kTMU: 64, 32, 16 or 8): every estimator matrix is read once per kTMU parameters.
// 32 when two CTAs of that size fit one SM, else the largest that fits (3D neighbourhoods with N = 40: 16).
// shared row stride kTMU + 4 (doubles): 4 or 12 mod 16 -> conflict-free DMMA fragment loads
constexpr int kTMUMax = 64;
constexpr int kMaxEstTerms = 64; // terms per subdomain

struct DevTerm {
  const double* M;
  int32_t rows, cols, left_kind, right_kind, qa, qb, out_kind, pad;
  double coef;
};

struct EstParams {
  int32_t n_sub, n_red, Q, n_theta, dmax_pad, qdmax_pad;
  const int32_t* offsets;     // n_sub + 1
  const int32_t* nbh_ptr;
  const int32_t* nbh_idx;
  const int32_t* term_ptr;    // n_sub + 1
  const DevTerm* terms;
  const double* rf2;
  const double* r_scale;
};

template <int kTMU>
__global__ void __launch_bounds__(kEstThreads, (kTMU <= 32) ? 2 : 1)
estimate_kernel(EstParams P, int64_t n_mu, const double* __restrict__ theta, const double* __restrict__ u,
                double* __restrict__ parts) {
  constexpr int kLDX = kTMU + 4;
  extern __shared__ double smem[];
  // Four spare rows behind each array: a term whose vector is a slice (u_i starts at row lo_self, any alignment) runs its
  // k loop to the next multiple of 4 and may read up to three rows past the neighbourhood's last; every row up to the end
  // of the arrays is zero-filled below, so 0 * (stale shared memory, possibly NaN / Inf) cannot reach a DMMA.
  double* XN = smem;                                   // (dmax_pad + 4) x kLDX
  double* XR = XN + (int64_t)(P.dmax_pad + 4) * kLDX;  // (qdmax_pad + 4) x kLDX
  double* TH = XR + (int64_t)(P.qdmax_pad + 4) * kLDX; // Q x kTMU
  double* OUTW = TH + P.Q * kTMU;                      // kEstWarps x 3 x kTMU
  __shared__ int s_tile_ptr[kMaxEstTerms + 1];         // row tiles (8 rows) of the subdomain's terms, prefix sums

  const int sub = blockIdx.y;
  const int64_t mu0 = (int64_t)blockIdx.x * kTMU;
  const int nmu = (int)min((int64_t)kTMU, n_mu - mu0);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;

  // ---- stage theta, u over the neighbourhood (dof-major in shared memory), and U_r = [theta_q u_k]
  for (int i = threadIdx.x; i < P.Q * kTMU; i += kEstThreads) {
    const int q = i / kTMU, m = i - q * kTMU;
    TH[i] = (m < nmu) ? theta[(mu0 + m) * P.n_theta + q] : 0.0;
  }
  for (int i = threadIdx.x; i < kEstWarps * 3 * kTMU; i += kEstThreads) OUTW[i] = 0.0;
  const int t0 = P.term_ptr[sub], n_terms = P.term_ptr[sub + 1] - t0;
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int k = 0; k < n_terms; ++k) { s_tile_ptr[k] = acc; acc += (P.terms[t0 + k].rows + 7) >> 3; }
    s_tile_ptr[n_terms] = acc;
  }
  const int nb0 = P.nbh_ptr[sub], nb1 = P.nbh_ptr[sub + 1];
  int d = 0, lo_self = 0;
  for (int e = nb0; e < nb1; ++e) {
    const int k = P.nbh_idx[e];
    const int off = P.offsets[k], Nk = P.offsets[k + 1] - off;
    if (k == sub) lo_self = d;
    for (int i = threadIdx.x; i < Nk * kTMU; i += kEstThreads) {
      const int m = i / Nk, a = i - m * Nk;
      XN[(d + a) * kLDX + m] = (m < nmu) ? u[(mu0 + m) * P.n_red + off + a] : 0.0;
    }
    d += Nk;
  }
  for (int i = threadIdx.x; i < (P.dmax_pad + 4 - d) * kTMU; i += kEstThreads) XN[(d + i / kTMU) * kLDX + (i % kTMU)] = 0.0;
  __syncthreads();
  {
    int lo = 0;
    for (int e = nb0; e < nb1; ++e) {
      const int k = P.nbh_idx[e];
      const int Nk = P.offsets[k + 1] - P.offsets[k];
      for (int i = threadIdx.x; i < P.Q * Nk * kTMU; i += kEstThreads) {
        const int m = i % kTMU, qa = i / kTMU;      // qa = q * Nk + a
        const int q = qa / Nk, a = qa - q * Nk;
        XR[(P.Q * lo + qa) * kLDX + m] = TH[q * kTMU + m] * XN[(lo + a) * kLDX + m];
      }
      lo += Nk;
    }
    const int qd = P.Q * d;
    for (int i = threadIdx.x; i < (P.qdmax_pad + 4 - qd) * kTMU; i += kEstThreads) XR[(qd + i / kTMU) * kLDX + (i % kTMU)] = 0.0;
  }
  __syncthreads();

  // ---- (term, 8-row tile) work items dealt round-robin to the warps: Y = M X on DMMA, then the column dot with X_L
  const int n_tiles = s_tile_ptr[n_terms];
  int ti = 0;
  for (int idx = warp; idx < n_tiles; idx += kEstWarps) {
    while (s_tile_ptr[ti + 1] <= idx) ++ti;
    const DevTerm T = P.terms[t0 + ti];
    const int r0 = 8 * (idx - s_tile_ptr[ti]);
    const double* XRt = (T.right_kind == LRBMS_VEC_UR) ? XR : (T.right_kind == LRBMS_VEC_UN ? XN : XN + lo_self * kLDX);
    const double* XLt = (T.left_kind == LRBMS_VEC_UR) ? XR : (T.left_kind == LRBMS_VEC_UN ? XN : XN + lo_self * kLDX);
    const int kend = (T.cols + 3) & ~3;
    double acc[kTMU / 8][2];
#pragma unroll
    for (int n = 0; n < kTMU / 8; ++n) acc[n][0] = acc[n][1] = 0.0;
    const bool rok = r0 + g < T.rows;
    const double* __restrict__ Mr = T.M + (int64_t)(r0 + g) * T.cols;
#pragma unroll 2
    for (int k0 = 0; k0 < kend; k0 += 4) {
      const double a = (rok && k0 + t < T.cols) ? __ldg(Mr + k0 + t) : 0.0;
      const double* xb = XRt + (k0 + t) * kLDX + g;
#pragma unroll
      for (int n = 0; n < kTMU / 8; ++n) dmma884(acc[n][0], acc[n][1], a, xb[8 * n]);
    }
    // column dot with the left vector (rows r0 + g, parameters 8n + 2t, 8n + 2t + 1), reduced over the 8 rows of the
    // tile (lanes with equal t), scaled, accumulated in this warp's private slice
#pragma unroll
    for (int n = 0; n < kTMU / 8; ++n) {
      double l0 = 0.0, l1 = 0.0;
      if (rok) {
        if (T.left_kind == LRBMS_VEC_ONE) { l0 = 1.0; l1 = 1.0; }
        else { l0 = XLt[(r0 + g) * kLDX + 8 * n + 2 * t]; l1 = XLt[(r0 + g) * kLDX + 8 * n + 2 * t + 1]; }
      }
      double v0 = l0 * acc[n][0], v1 = l1 * acc[n][1];
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {
        v0 += __shfl_xor_sync(0xffffffffu, v0, o);
        v1 += __shfl_xor_sync(0xffffffffu, v1, o);
      }
      if (g == 0) {
        const int m = 8 * n + 2 * t;
        double cf0 = T.coef, cf1 = T.coef;
        if (T.qa >= 0) { cf0 *= TH[T.qa * kTMU + m]; cf1 *= TH[T.qa * kTMU + m + 1]; }
        if (T.qb >= 0) { cf0 *= TH[T.qb * kTMU + m]; cf1 *= TH[T.qb * kTMU + m + 1]; }
        OUTW[(warp * 3 + T.out_kind) * kTMU + m] += cf0 * v0;
        OUTW[(warp * 3 + T.out_kind) * kTMU + m + 1] += cf1 * v1;
      }
    }
    __syncwarp();
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * kTMU; i += kEstThreads) {
    const int kind = i / kTMU, m = i - kind * kTMU;
    if (m >= nmu) continue;
    double v = 0.0;
    for (int w = 0; w < kEstWarps; ++w) v += OUTW[(w * 3 + kind) * kTMU + m];
    if (kind == LRBMS_OUT_R) v = (P.rf2[sub] + v) * P.r_scale[sub];
    parts[((int64_t)kind * P.n_sub + sub) * n_mu + mu0 + m] = v;
  }
}

struct CombineParams {
  int32_t n_sub, Q, n_theta, alpha_first;
  double theta_bar[16], theta_hat[16];
};

// eta = ( sqrt(gamma) ||nc||_2 + ||r + df||_2 / sqrt(alpha_hat) ) / sqrt(alpha_bar)       (estimators.py:99-102),
// norms over subdomains per parameter column (SURVEY.md 8a a14 quirk 4); optional indicators (estimators.py:104-109)
__global__ void combine_kernel(CombineParams P, int64_t n_mu, const double* __restrict__ theta,
                               const double* __restrict__ parts, double* __restrict__ eta, double* __restrict__ indicators) {
  const int64_t mu = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (mu >= n_mu) return;
  double a_bar = INFINITY, a_hat = INFINITY, g_bar = -INFINITY;
  for (int q = 0; q < P.Q; ++q) {
    const double th = theta[mu * P.n_theta + q];
    const double rb = th / P.theta_bar[q], rh = th / P.theta_hat[q];
    if (!(P.alpha_first && q > 0)) { a_bar = fmin(a_bar, rb); a_hat = fmin(a_hat, rh); }
    g_bar = fmax(g_bar, rb);
  }
  double snc = 0.0, srd = 0.0;
  const double* nc = parts;
  const double* r = parts + (int64_t)P.n_sub * n_mu;
  const double* df = parts + 2 * (int64_t)P.n_sub * n_mu;
  for (int i = 0; i < P.n_sub; ++i) {
    const double a = nc[i * n_mu + mu], b = r[i * n_mu + mu] + df[i * n_mu + mu];
    snc += a * a;
    srd += b * b;
    if (indicators) indicators[i * n_mu + mu] = (2.0 / a_bar) * (g_bar * a * a + (1.0 / a_hat) * b * b);
  }
  eta[mu] = (sqrt(g_bar) * sqrt(snc) + sqrt(srd) / sqrt(a_hat)) / sqrt(a_bar);
}

__global__ void eta_max_kernel(int64_t n, const double* __restrict__ eta, double* __restrict__ max_out,
                               int64_t* __restrict__ arg_out) {
  __shared__ double sv[1024];
  __shared__ int64_t si[1024];
  double best = -INFINITY;
  int64_t bi = -1;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = eta[i];
    if (v > best || bi < 0) { best = v; bi = i; }
  }
  sv[threadIdx.x] = best;
  si[threadIdx.x] = bi;
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      const double v = sv[threadIdx.x + s];
      const int64_t j = si[threadIdx.x + s];
      if (j >= 0 && (si[threadIdx.x] < 0 || v > sv[threadIdx.x] || (v == sv[threadIdx.x] && j < si[threadIdx.x]))) {
        sv[threadIdx.x] = v;
        si[threadIdx.x] = j;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { *max_out = sv[0]; *arg_out = si[0]; }
}

// ------------------------------------------------------------------------------------------------------
//  plan
// ------------------------------------------------------------------------------------------------------
struct OnlinePlan : lrbms_plan {
  lrbms_symbolic sym;
  // selected solve kernel: LRBMS_SOLVER_WINDOW (solve_kernel_v2) or LRBMS_SOLVER_BANDED (band.cu: block-banded
  // out-of-HBM Cholesky for systems whose factor window exceeds one SM)
  int solver = LRBMS_SOLVER_AUTO;
  SolveParamsV2 sp2;
  lrbms_band_plan band;
  int64_t solve_stride = 0;     // doubles of factor scratch per resident CTA of the window kernel
  EstParams ep;
  CombineParams cp;
  int solve_grid = 0;
  size_t solve_smem = 0, est_smem = 0;
  int est_tmu = kTMUMax;        // parameters per estimator CTA
  bool has_estimator = false;
  int run(void*) override { return lrbms_fail(ctx, LRBMS_ERR_INVALID, "online plans are run with lrbms_online_*"); }
  ~OnlinePlan() override { lrbms_band_release(band); }
};

}  // namespace

extern "C" {

int lrbms_online_plan_create(lrbms_handle_t h, const lrbms_reduced_system_t* sys, lrbms_plan_t* out) {
  LRBMS_REQUIRE(h, h && sys && out, "online_plan_create: null argument");
  LRBMS_REQUIRE(h, sys->Q >= 1 && sys->Q <= 16 && sys->Qf >= 1 && sys->Qf <= 16, "online_plan_create: 1 <= Q, Qf <= 16");
  LRBMS_REQUIRE(h, sys->lhs_blocks && sys->rhs && sys->block_offset && sys->basis_sizes, "online_plan_create: null data pointer");
  LRBMS_REQUIRE(h, sys->solver == LRBMS_SOLVER_AUTO || sys->solver == LRBMS_SOLVER_WINDOW || sys->solver == LRBMS_SOLVER_BANDED,
                "online_plan_create: unknown solver");
  LRBMS_CUDA_CHECK(h, cudaSetDevice(h->device));
  OnlinePlan* P = new OnlinePlan();
  P->ctx = h;
  P->kind = PLAN_ONLINE;
  std::string err;
  int rc = lrbms_symbolic_basics(P->sym, sys->n_sub, sys->basis_sizes, sys->n_blocks, sys->block_i, sys->block_j, &err);
  if (rc) { delete P; return lrbms_fail(h, rc, err); }
  // The 8x8-tile schedule is only built when the window kernel can use it: its pair lists grow like
  // n (b / 8)^2 / 2 (135 M pairs for the 8x8x8, N = 40 system), the band solver needs none of it.
  const double est_pairs = 0.5 * P->sym.ntc * (P->sym.half_bandwidth / 8.0 + 1.0) * (P->sym.half_bandwidth / 8.0 + 1.0);
  const bool tiles_built = sys->solver == LRBMS_SOLVER_WINDOW || (sys->solver == LRBMS_SOLVER_AUTO && est_pairs <= 3.0e7);
  if (tiles_built) {
    rc = lrbms_symbolic_build(P->sym, sys->n_sub, sys->basis_sizes, sys->n_blocks, sys->block_i, sys->block_j, &err);
    if (rc) { delete P; return lrbms_fail(h, rc, err); }
  }
  const lrbms_symbolic& S = P->sym;
  const int Q = sys->Q, Qf = sys->Qf;

  // ---- download the reduced blocks and the rhs
  int64_t n_doubles = 0;
  for (int q = 0; q < Q; ++q)
    for (int b = 0; b < sys->n_blocks; ++b)
      n_doubles = std::max<int64_t>(n_doubles, sys->block_offset[(int64_t)q * sys->n_blocks + b] +
                                                   (int64_t)S.sizes[sys->block_i[b]] * S.sizes[sys->block_j[b]]);
  std::vector<double> hb((size_t)std::max<int64_t>(1, n_doubles));
  if (n_doubles) {
    cudaError_t e = cudaMemcpy(hb.data(), sys->lhs_blocks, sizeof(double) * n_doubles, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { delete P; return lrbms_fail(h, LRBMS_ERR_CUDA, cudaGetErrorString(e)); }
  }
  std::vector<double> tmp((size_t)Qf * S.n_red);     // [Qf][n_red], as given
  {
    cudaError_t e = cudaMemcpy(tmp.data(), sys->rhs, sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { delete P; return lrbms_fail(h, LRBMS_ERR_CUDA, cudaGetErrorString(e)); }
  }

// CUDA calls after the plan object exists: destroy it on failure (no leaked plans on error paths)
#define PLAN_CUDA_CHECK(expr)                                                                          \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess) {                                                                           \
      lrbms_plan_destroy(P);                                                                           \
      return lrbms_fail(h, LRBMS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));        \
    }                                                                                                  \
  } while (0)
  int32_t *d_i32 = nullptr;
  double* d_f64 = nullptr;
#define UP_I32(field, vec) do { rc = plan_upload(P, &d_i32, vec); if (rc) { lrbms_plan_destroy(P); return rc; } field = d_i32; } while (0)
#define UP_F64(field, vec) do { rc = plan_upload(P, &d_f64, vec); if (rc) { lrbms_plan_destroy(P); return rc; } field = d_f64; } while (0)
  // ---- shared-memory-window kernel: used whenever the live window of L fits into the shared memory of one SM
  if (tiles_built) {
    size_t static2 = 0;
    PLAN_CUDA_CHECK(lrbms_open_dynamic_smem(h, (const void*)solve_kernel_v2, &static2));
    // the static shared memory of the kernel (mbarriers, status word) counts against the same per-block limit
    const int64_t smem_budget = (int64_t)h->max_smem_optin - (int64_t)static2;
    if ((int64_t)lrbms_window_smem_bytes(S, Q) <= smem_budget) {
      // The window kernel runs; factor in the subdomain order its cost model prefers (within the same shared memory).
      rc = lrbms_symbolic_choose_order(P->sym, Q, smem_budget, &err);
      if (rc) { lrbms_plan_destroy(P); return lrbms_fail(h, rc, err); }
      const int maxcol = std::max(1, S.max_targets - 1);
      const int MT = S.max_targets;
      const int64_t region = std::max<int64_t>((int64_t)S.n_win_slots * 64, (int64_t)kBackStages * maxcol * 64);
      const int mcp = std::max(1, S.max_col_pairs);
      // operator tiles of the permuted system: the lower triangle of every stored block (i >= j) goes to its permuted
      // rows and columns, transposed where the order puts subdomain j after subdomain i
      std::vector<double> tiles((size_t)Q * S.n_a_tiles * 64, 0.0);
      auto slot_of = [&](int I, int J) {
        const int32_t* b = S.row_idx.data() + S.col_ptr[J];
        const int32_t* e = S.row_idx.data() + S.col_ptr[J + 1];
        return (int32_t)(std::lower_bound(b, e, I) - S.row_idx.data());
      };
      for (int q = 0; q < Q; ++q)
        for (int b = 0; b < sys->n_blocks; ++b) {
          const int i = sys->block_i[b], j = sys->block_j[b];
          if (i < j) continue;
          const double* blk = hb.data() + sys->block_offset[(int64_t)q * sys->n_blocks + b];
          const int Ni = S.sizes[i], Nj = S.sizes[j];
          const bool flip = S.iperm[i] < S.iperm[j];
          for (int a = 0; a < Ni; ++a)
            for (int c = 0; c < Nj; ++c) {
              int r = S.perm_offsets[i] + a, cc = S.perm_offsets[j] + c;
              if (flip) std::swap(r, cc);
              if (r < cc) continue;
              const int ai = S.a_map[slot_of(r / 8, cc / 8)];
              double* tl = tiles.data() + ((size_t)q * S.n_a_tiles + ai) * 64;
              tl[(r & 7) * 8 + (cc & 7)] = blk[(int64_t)a * Nj + c];
              if (r / 8 == cc / 8) tl[(cc & 7) * 8 + (r & 7)] = blk[(int64_t)a * Nj + c];
            }
        }
      std::vector<double> rhs_h((size_t)Qf * S.n_pad, 0.0);
      for (int q = 0; q < Qf; ++q)
        for (int r = 0; r < S.n_red; ++r) rhs_h[(size_t)q * S.n_pad + r] = tmp[(size_t)q * S.n_red + S.row_map[r]];
      SolveParamsV2& s2 = P->sp2;
      s2.n_red = S.n_red; s2.n_pad = S.n_pad; s2.ntc = S.ntc; s2.Q = Q; s2.Qf = Qf; s2.n_theta = Q + Qf;
      s2.n_a_tiles = S.n_a_tiles;
      s2.work_stride = (int64_t)S.n_tiles() * 64;
      UP_I32(s2.row_idx, S.row_idx);
      UP_I32(s2.row_map, S.row_map);
      UP_F64(s2.a_tiles, tiles);
      UP_F64(s2.rhs, rhs_h);
      s2.region_doubles = (int32_t)region;
      s2.max_targets = MT;
      s2.max_col_pairs = mcp;
      s2.a_ring = S.a_ring;
      s2.back_stage_doubles = maxcol * 64;
      s2.n_ca = (int32_t)S.ca_tile.size();
      UP_I32(s2.cslot, S.cslot);
      UP_I32(s2.cord, S.cord);
      UP_I32(s2.cnext, S.cnext);
      UP_I32(s2.ca_tile, S.ca_tile);
      const int32_t* tmp = nullptr;
      UP_I32(tmp, S.ccol);   s2.ccol = reinterpret_cast<const int4*>(tmp);
      UP_I32(tmp, S.cinfo);  s2.ccol2 = reinterpret_cast<const int4*>(tmp);
      UP_I32(tmp, S.ccol3);  s2.ccol3 = reinterpret_cast<const int4*>(tmp);
      UP_I32(tmp, S.cdesc);  s2.cdesc = reinterpret_cast<const int4*>(tmp);
      UP_I32(tmp, S.win_ab); s2.win_ab = reinterpret_cast<const int2*>(tmp);
      s2.staggered = S.staggered;
#ifdef LRBMS_DEVTOOLS
      s2.timing = nullptr;
      if (const char* tenv = getenv("LRBMS_SOLVE_TIMING")) {
        if (atoi(tenv) > 0) {
          rc = plan_alloc(P, &s2.timing, (size_t)kV2Warps * 8);
          if (rc) { lrbms_plan_destroy(P); return rc; }
          PLAN_CUDA_CHECK(cudaMemset(s2.timing, 0, sizeof(long long) * kV2Warps * 8));
        }
      }
#endif
      P->solve_smem = lrbms_window_smem_bytes(S, Q);
      P->solver = LRBMS_SOLVER_WINDOW;
      P->solve_grid = h->sm_count;
      P->solve_stride = s2.work_stride;
    }
  }
  if (sys->solver == LRBMS_SOLVER_WINDOW && P->solver != LRBMS_SOLVER_WINDOW) {
    lrbms_plan_destroy(P);
    return lrbms_fail(h, LRBMS_ERR_UNSUPPORTED, "online_plan_create: the live factor window does not fit the shared memory of one SM");
  }
  // ---- band solver (band.cu): everything the CTA-per-parameter window kernel cannot hold
  if (P->solver != LRBMS_SOLVER_WINDOW) {
    rc = lrbms_band_build(P, P->band, S.n_sub, S.sizes.data(), S.offsets.data(), Q, Qf, sys->n_blocks, sys->block_i, sys->block_j,
                          sys->block_offset, hb.data(), tmp.data());
    if (rc) { lrbms_plan_destroy(P); return rc; }
    P->solver = LRBMS_SOLVER_BANDED;
    P->solve_grid = h->sm_count;
  }

  // ---- estimator tables
  P->has_estimator = sys->n_terms > 0;
  if (P->has_estimator) {
    if (!(sys->nbh_ptr && sys->nbh_idx && sys->terms && sys->est_matrices && sys->rf_squared && sys->r_scale &&
          sys->theta_bar && sys->theta_hat)) {
      lrbms_plan_destroy(P);
      return lrbms_fail(h, LRBMS_ERR_INVALID, "online_plan_create: estimator data missing");
    }
    EstParams& ep = P->ep;
    ep.n_sub = S.n_sub; ep.n_red = S.n_red; ep.Q = Q; ep.n_theta = Q + Qf;
    std::vector<int32_t> nbh_ptr(sys->nbh_ptr, sys->nbh_ptr + S.n_sub + 1);
    std::vector<int32_t> nbh_idx(sys->nbh_idx, sys->nbh_idx + nbh_ptr[S.n_sub]);
    int dmax = 0;
    std::vector<int> dsub(S.n_sub, 0);
    for (int i = 0; i < S.n_sub; ++i) {
      int d = 0;
      bool self = false;
      for (int e = nbh_ptr[i]; e < nbh_ptr[i + 1]; ++e) {
        const int k = nbh_idx[e];
        if (k < 0 || k >= S.n_sub) { lrbms_plan_destroy(P); return lrbms_fail(h, LRBMS_ERR_INVALID, "online_plan_create: neighbourhood index out of range"); }
        d += S.sizes[k];
        self |= (k == i);
      }
      if (!self) { lrbms_plan_destroy(P); return lrbms_fail(h, LRBMS_ERR_INVALID, "online_plan_create: neighbourhood must contain the subdomain itself"); }
      dsub[i] = d;
      dmax = std::max(dmax, d);
    }
    ep.dmax_pad = (dmax + 3) & ~3;
    ep.qdmax_pad = (Q * dmax + 3) & ~3;
    // sort terms by subdomain, validate shapes
    std::vector<std::vector<DevTerm>> per_sub(S.n_sub);
    for (int k = 0; k < sys->n_terms; ++k) {
      const lrbms_estimator_term_t& T = sys->terms[k];
      bool ok = T.subdomain >= 0 && T.subdomain < S.n_sub && T.out_kind >= 0 && T.out_kind < 3 && T.qa < Q && T.qb < Q;
      auto dim_of = [&](int kind, int i) { return kind == LRBMS_VEC_ONE ? 1 : kind == LRBMS_VEC_UI ? S.sizes[i] : kind == LRBMS_VEC_UN ? dsub[i] : Q * dsub[i]; };
      if (ok) ok = T.rows == dim_of(T.left_kind, T.subdomain) && T.cols == dim_of(T.right_kind, T.subdomain) && T.right_kind != LRBMS_VEC_ONE;
      if (!ok) { lrbms_plan_destroy(P); return lrbms_fail(h, LRBMS_ERR_INVALID, "online_plan_create: estimator term " + std::to_string(k) + " is inconsistent"); }
      DevTerm D;
      D.M = sys->est_matrices + T.matrix_offset; D.rows = T.rows; D.cols = T.cols; D.left_kind = T.left_kind;
      D.right_kind = T.right_kind; D.qa = T.qa; D.qb = T.qb; D.out_kind = T.out_kind; D.pad = 0; D.coef = T.coef;
      per_sub[T.subdomain].push_back(D);
    }
    std::vector<int32_t> term_ptr(S.n_sub + 1, 0);
    std::vector<DevTerm> terms;
    double est_flops = 0;
    for (int i = 0; i < S.n_sub; ++i) {
      if ((int)per_sub[i].size() > kMaxEstTerms) {
        lrbms_plan_destroy(P);
        return lrbms_fail(h, LRBMS_ERR_UNSUPPORTED, "online_plan_create: more than 64 estimator terms on one subdomain");
      }
      for (const DevTerm& D : per_sub[i]) { terms.push_back(D); est_flops += 2.0 * D.rows * D.cols; }
      term_ptr[i + 1] = (int32_t)terms.size();
    }
    P->info_flops = est_flops;   // estimator flops per mu (factor flops are in lrbms_symbolic_info)
    UP_I32(ep.offsets, S.offsets);
    UP_I32(ep.nbh_ptr, nbh_ptr);
    UP_I32(ep.nbh_idx, nbh_idx);
    UP_I32(ep.term_ptr, term_ptr);
    DevTerm* d_terms = nullptr;
    rc = plan_upload(P, &d_terms, terms);
    if (rc) { lrbms_plan_destroy(P); return rc; }
    ep.terms = d_terms;
    std::vector<double> rf2(sys->rf_squared, sys->rf_squared + S.n_sub), rs(sys->r_scale, sys->r_scale + S.n_sub);
    UP_F64(ep.rf2, rf2);
    UP_F64(ep.r_scale, rs);
    auto est_bytes = [&](int tmu) {
      return sizeof(double) * ((size_t)(ep.dmax_pad + ep.qdmax_pad + 8) * (tmu + 4) + (size_t)Q * tmu + kEstWarps * 3 * tmu);
    };
    // dynamic bytes each instantiation may ask for: the per-block limit minus its static shared memory (s_tile_ptr)
    auto est_room = [&](int tmu, size_t* room) {
      const void* fn = tmu == 64 ? (const void*)estimate_kernel<64>
                       : tmu == 32 ? (const void*)estimate_kernel<32>
                       : tmu == 16 ? (const void*)estimate_kernel<16> : (const void*)estimate_kernel<8>;
      size_t st = 0;
      const cudaError_t e = lrbms_open_dynamic_smem(h, fn, &st);
      *room = (size_t)h->max_smem_optin - st;
      return e;
    };
    // 32 parameters per CTA when two such CTAs fit one SM (the staging phase of one overlaps the DMMAs of the other:
    // 4.5 instead of 5.4 ms per 10 000 parameters at C2), else the largest tile that fits at all
    P->est_tmu = (2 * (est_bytes(32) + 1024) <= (size_t)h->max_smem_optin) ? 32 : kTMUMax;
    size_t room = 0;
    PLAN_CUDA_CHECK(est_room(P->est_tmu, &room));
    while (P->est_tmu > 8 && est_bytes(P->est_tmu) > room) {
      P->est_tmu /= 2;
      PLAN_CUDA_CHECK(est_room(P->est_tmu, &room));
    }
    P->est_smem = est_bytes(P->est_tmu);
    if (P->est_smem > room) {
      lrbms_plan_destroy(P);
      return lrbms_fail(h, LRBMS_ERR_UNSUPPORTED, "online_plan_create: neighbourhood too large for the estimator kernel's shared memory");
    }
    CombineParams& cp = P->cp;
    cp.n_sub = S.n_sub; cp.Q = Q; cp.n_theta = Q + Qf; cp.alpha_first = sys->alpha_returns_first;
    for (int q = 0; q < Q; ++q) { cp.theta_bar[q] = sys->theta_bar[q]; cp.theta_hat[q] = sys->theta_hat[q]; }
  }
#undef UP_I32
#undef UP_F64
  P->info_launches = P->solver == LRBMS_SOLVER_BANDED ? 4.0 * P->band.nbc + 4 : 3;
  P->info_ctas = P->solve_grid;
  // introspection (lrbms_plan_info 6 .. 9): which solve kernel the plan selected, executed factor flops per parameter
  // (the 8x8-tile count for the window kernel, the dense-band count of the band solver), half bandwidth,
  // parameters per estimator CTA
  P->info_solver = P->solver;
  P->info_solve_flops = P->solver == LRBMS_SOLVER_BANDED ? P->band.flops_per_mu : (double)S.flops;
  P->info_half_bandwidth = S.half_bandwidth;
  P->info_est_tmu = P->has_estimator ? P->est_tmu : 0;
  // uploads and clears above ran on the legacy default stream: finish them before a caller's non-blocking stream runs the plan
  PLAN_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)0));
  *out = P;
  return LRBMS_OK;
}

static size_t solve_ws_bytes(const OnlinePlan* P, int64_t n_mu) {
  if (P->solver == LRBMS_SOLVER_BANDED) return lrbms_band_workspace_bytes(P->band, n_mu);
  const int64_t ctas = std::min<int64_t>(P->solve_grid, std::max<int64_t>(1, n_mu));
  return (size_t)ctas * P->solve_stride * sizeof(double);
}
static size_t parts_ws_bytes(const OnlinePlan* P, int64_t n_mu) {
  return (size_t)3 * P->sym.n_sub * std::max<int64_t>(1, n_mu) * sizeof(double);
}

int lrbms_online_workspace_bytes(lrbms_plan_t plan, int64_t n_mu, size_t* bytes) {
  if (!plan || plan->kind != PLAN_ONLINE || !bytes) return LRBMS_ERR_INVALID;
  const OnlinePlan* P = static_cast<const OnlinePlan*>(plan);
  *bytes = ((solve_ws_bytes(P, n_mu) + 255) & ~(size_t)255) + parts_ws_bytes(P, n_mu);
  return LRBMS_OK;
}

int lrbms_online_solve(lrbms_plan_t plan, int64_t n_mu, const double* theta, double* u, int32_t* info, void* workspace,
                       size_t workspace_bytes, void* stream) {
  if (!plan || plan->kind != PLAN_ONLINE) return LRBMS_ERR_INVALID;
  OnlinePlan* P = static_cast<OnlinePlan*>(plan);
  LRBMS_REQUIRE(P->ctx, theta && u && workspace, "online_solve: null argument");
  if (n_mu <= 0) return LRBMS_OK;
  if (P->solver == LRBMS_SOLVER_BANDED) {
    // the band solver works through the batch in chunks of as many parameters as the workspace holds factors for
    LRBMS_REQUIRE(P->ctx, lrbms_band_chunk(P->band, n_mu, workspace_bytes) >= 1,
                  "online_solve: workspace too small (see lrbms_online_workspace_bytes)");
    return lrbms_band_solve(P->ctx, P->band, n_mu, theta, u, info, workspace, solve_ws_bytes(P, n_mu) <= workspace_bytes
                            ? solve_ws_bytes(P, n_mu) : workspace_bytes, (cudaStream_t)stream);
  }
  LRBMS_REQUIRE(P->ctx, workspace_bytes >= solve_ws_bytes(P, n_mu), "online_solve: workspace too small (see lrbms_online_workspace_bytes)");
  const int grid = (int)std::min<int64_t>(P->solve_grid, n_mu);
  solve_kernel_v2<<<grid, kV2Threads, P->solve_smem, (cudaStream_t)stream>>>(P->sp2, n_mu, theta, u, info, (double*)workspace);
  LRBMS_CUDA_CHECK(P->ctx, cudaGetLastError());
  return LRBMS_OK;
}

int lrbms_online_estimate(lrbms_plan_t plan, int64_t n_mu, const double* theta, const double* u, double* eta, double* parts,
                          double* indicators, void* workspace, size_t workspace_bytes, void* stream) {
  if (!plan || plan->kind != PLAN_ONLINE) return LRBMS_ERR_INVALID;
  OnlinePlan* P = static_cast<OnlinePlan*>(plan);
  LRBMS_REQUIRE(P->ctx, P->has_estimator, "online_estimate: the plan was created without estimator terms");
  LRBMS_REQUIRE(P->ctx, theta && u && eta, "online_estimate: null argument");
  if (n_mu <= 0) return LRBMS_OK;
  double* pbuf = parts;
  if (!pbuf) {
    const size_t off = (solve_ws_bytes(P, n_mu) + 255) & ~(size_t)255;
    LRBMS_REQUIRE(P->ctx, workspace && workspace_bytes >= off + parts_ws_bytes(P, n_mu), "online_estimate: workspace too small");
    pbuf = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + off);
  }
  const int tmu = P->est_tmu;
  dim3 grid((unsigned)((n_mu + tmu - 1) / tmu), (unsigned)P->sym.n_sub);
  cudaStream_t es = (cudaStream_t)stream;
  if (tmu == 64) estimate_kernel<64><<<grid, kEstThreads, P->est_smem, es>>>(P->ep, n_mu, theta, u, pbuf);
  else if (tmu == 32) estimate_kernel<32><<<grid, kEstThreads, P->est_smem, es>>>(P->ep, n_mu, theta, u, pbuf);
  else if (tmu == 16) estimate_kernel<16><<<grid, kEstThreads, P->est_smem, es>>>(P->ep, n_mu, theta, u, pbuf);
  else estimate_kernel<8><<<grid, kEstThreads, P->est_smem, es>>>(P->ep, n_mu, theta, u, pbuf);
  combine_kernel<<<(unsigned)((n_mu + 127) / 128), 128, 0, (cudaStream_t)stream>>>(P->cp, n_mu, theta, pbuf, eta, indicators);
  LRBMS_CUDA_CHECK(P->ctx, cudaGetLastError());
  return LRBMS_OK;
}

int lrbms_online_sweep(lrbms_plan_t plan, int64_t n_mu, const double* theta, double* u, double* eta, double* parts,
                       double* indicators, int32_t* info, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = lrbms_online_solve(plan, n_mu, theta, u, info, workspace, workspace_bytes, stream);
  if (rc) return rc;
  return lrbms_online_estimate(plan, n_mu, theta, u, eta, parts, indicators, workspace, workspace_bytes, stream);
}

int lrbms_online_debug_timing(lrbms_plan_t plan, int64_t* out_host, int32_t n) {
  if (!plan || plan->kind != PLAN_ONLINE || !out_host) return LRBMS_ERR_INVALID;
  OnlinePlan* P = static_cast<OnlinePlan*>(plan);
#ifdef LRBMS_DEVTOOLS
  long long* src = P->solver == LRBMS_SOLVER_WINDOW ? P->sp2.timing : nullptr;
  if (!src) return lrbms_fail(P->ctx, LRBMS_ERR_INVALID, "debug timing is off (set LRBMS_SOLVE_TIMING=1 before creating the plan)");
  const int cnt = std::min<int>(n, kV2Warps * 8);
  LRBMS_CUDA_CHECK(P->ctx, cudaMemcpy(out_host, src, sizeof(long long) * cnt, cudaMemcpyDeviceToHost));
  return cnt;
#else
  (void)n;
  return lrbms_fail(P->ctx, LRBMS_ERR_UNSUPPORTED, "debug timing needs a developer build of the library (-DLRBMS_DEVTOOLS)");
#endif
}

int lrbms_eta_max(lrbms_handle_t h, int64_t n_mu, const double* eta, double* max_out, int64_t* argmax_out, void* stream) {
  LRBMS_REQUIRE(h, h && eta && max_out && argmax_out && n_mu > 0, "eta_max: bad argument");
  eta_max_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(n_mu, eta, max_out, argmax_out);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  return LRBMS_OK;
}

}  // extern "C"
