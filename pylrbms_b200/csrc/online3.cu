// solve_kernel_v3: the shared-memory-window tile Cholesky of online.cu processed in PANELS of two tile columns.
//
// replaces (like solve_kernel_v2): LincombOperator.assemble(mu) + numpy.linalg.solve on the unblocked reduced operator behind
// rd.solve(mu) (reference online_enrichment.py:72, scripts/online_adaptive_lrbms.py:141), one CTA per parameter.
//
// Why panels.  The one-column kernel multiplies one target tile by one operand tile from each side per step: two
// shared-memory fragment loads per two DMMAs, which is exactly the ratio at which the single shared-memory port of an SM
// saturates together with the FP64 tensor pipe (ncu: 614 k shared-memory wavefronts per parameter against 84 k DMMAs, the
// port 54 % busy, the pipe 30 %).  With two tile columns per panel every early-update step owns a 2 x 2 block of target tiles
// and loads two operand tiles from each side: four loads per eight DMMAs.  The fixed costs of a pipeline stage (solves of
// the finished panel, barriers) are paid once per two columns.
//
// Pipeline, iteration p (q = p + 1; tables from symbolic3.cpp, executed in NumPy by tests/test_symbolic3_emulator.py):
//   A   update warps 1..15: early updates of panel q (sources: every column before panel p) in 2 x 2 register blocks; long
//       blocks are cut into chunks, the extra chunks go to a partial buffer.  Warp 0 is still busy with the chain of panel p.
//   --- barrier (all)
//   B1  update warps: solve their rows of panel p against the diagonal block of panel p (X0 = C0 W00^T, X1 = (C1 - X0 L10^T)
//       W11^T), store them (window + factor), keep them as fragments.  Warp 0: the same for the two HEAD rows (the diagonal
//       rows of panel q), and the partial blocks of panel q's diagonal block.
//   --- barrier X (warp 0 only arrives)
//   B2  update warps: partial blocks + late update (sources: panel p) of their block of panel q, result to the accumulator
//       ring.  Warp 0: late update of the diagonal block, then the critical chain of panel q (two 8x8 Cholesky factorisations
//       and inverses, one tile solve, one tile update) -- it runs on while the others do A of the next iteration.
//   --- barrier (update warps)
// The forward substitution rides along as one more block; the backward substitution streams the factor back (bulk copies).
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "online3.h"

namespace {

constexpr int kThreads3 = kV3Warps * 32;
constexpr int kBack3 = 6;            // backward-substitution ring

__device__ __forceinline__ void bar_sync_named(int id, int count) { asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void bar_arrive_named(int id, int count) { asm volatile("bar.arrive %0, %1;\n" ::"r"(id), "r"(count) : "memory"); }

// acc (accumulator layout: lane (g, t) holds T[g][2t], T[g][2t+1]) -= A * B^T with A, B in operand-fragment order
__device__ __forceinline__ void tile_msub(double2& acc, const double2 fa, const double2 fb) {
  dmma884(acc.x, acc.y, -fa.x, fb.x);
  dmma884(acc.x, acc.y, -fa.y, fb.y);
}
// X = C * W^T: C as an A fragment, W row-major in shared memory
__device__ __forceinline__ double2 tile_times_wt(const double2 fc, const double* __restrict__ sWm, int g, int t) {
  double2 x = make_double2(0.0, 0.0);
  dmma884(x.x, x.y, fc.x, sWm[g * 8 + t]);
  dmma884(x.x, x.y, fc.y, sWm[g * 8 + 4 + t]);
  return x;
}
// accumulator layout -> operand fragment through a row-major scratch tile (one warp; the tile is dead afterwards)
__device__ __forceinline__ double2 to_fragment(double* scratch, const double2 x, int g, int t) {
  __syncwarp();
  *reinterpret_cast<double2*>(scratch + g * 8 + 2 * t) = x;
  __syncwarp();
  return make_double2(scratch[g * 8 + t], scratch[g * 8 + t + 4]);
}

// The two tiles of one row of panel p solved against the panel's diagonal block (sWp: W00, L10, W11 row-major).
// c0t / c1t: the row's accumulator tiles (row-major, also used as scratch).  Returns the two solved tiles as fragments; x0 / x1
// (accumulator layout) are what the forward-substitution block stores as y.
__device__ __forceinline__ void solve_row(double* c0t, double* c1t, const double* __restrict__ sWp, int g, int t, double2& f0,
                                          double2& f1, double2& x0, double2& x1) {
  const double2 a0 = make_double2(c0t[g * 8 + t], c0t[g * 8 + t + 4]);
  double2 c1 = *reinterpret_cast<const double2*>(c1t + g * 8 + 2 * t);
  x0 = tile_times_wt(a0, sWp, g, t);
  f0 = to_fragment(c0t, x0, g, t);
  tile_msub(c1, f0, make_double2(sWp[64 + g * 8 + t], sWp[64 + g * 8 + t + 4]));      // C1 -= X0 L10^T
  const double2 a1 = to_fragment(c1t, c1, g, t);
  x1 = tile_times_wt(a1, sWp + 128, g, t);
  f1 = to_fragment(c1t, x1, g, t);
}

// 8x8 Cholesky + inverse of a row-major tile in shared memory, redundantly per lane in registers (no cross-lane traffic on
// the critical chain).  Writes W = L^-1 row-major to sWout and to the factor's diagonal slot.  Returns the first bad pivot.
__device__ __forceinline__ int potrf_inverse(const double* __restrict__ tile, double* __restrict__ sWout, double* __restrict__ gout,
                                             int col0, int n_red, int lane) {
  double l[36], rinv[8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j <= i; ++j) l[i * (i + 1) / 2 + j] = tile[i * 8 + j];
  int bad = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    double akk = l[k * (k + 1) / 2 + k];
    if (col0 + k >= n_red) akk = 1.0;                    // padding rows: identity
    if (!(akk > 0.0)) { if (!bad) bad = col0 + k + 1; akk = 1.0; }
    const double r = rsqrt(akk);
    rinv[k] = r;
#pragma unroll
    for (int i = k + 1; i < 8; ++i) l[i * (i + 1) / 2 + k] *= r;
#pragma unroll
    for (int j = k + 1; j < 8; ++j)
#pragma unroll
      for (int i = j; i < 8; ++i) l[i * (i + 1) / 2 + j] -= l[i * (i + 1) / 2 + k] * l[j * (j + 1) / 2 + k];
  }
  const int c = lane & 7;
  double w[8];
#pragma unroll
  for (int ii = 0; ii < 8; ++ii) {
    double s = (ii == c) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 0; k < ii; ++k) s -= l[ii * (ii + 1) / 2 + k] * w[k];
    w[ii] = s * rinv[ii];
  }
  __syncwarp();
  if (lane < 8) {
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
      sWout[ii * 8 + c] = w[ii];
      gout[ii * 8 + c] = w[ii];
    }
  }
  __syncwarp();
  return bad;
}

__global__ void __launch_bounds__(kThreads3, 1)
solve_kernel_v3(V3Params P, int64_t n_mu, const double* __restrict__ theta, double* __restrict__ u, int32_t* __restrict__ info,
                double* __restrict__ work) {
  extern __shared__ __align__(16) double smem[];
  double* win = smem;                                          // region_doubles (window incl. the zero tile; backward ring)
  double* accbuf = win + P.region_doubles;                     // (2 acc_rows + 2) tiles, row-major
  double* part = accbuf + (2 * P.acc_rows + 2) * 64;           // n_partial blocks of 4 tiles
  double* sx = part + P.n_partial * 256;                       // n_pad
  double* sW = sx + P.n_pad;                                   // [2][3][64]: W00, L10, W11 of the even / odd panels
  double* sred = sW + 2 * 3 * 64;                              // 2 * 16 * 8 (backward substitution)
  double* sth = sred + 2 * kV3Warps * 8;                       // 32
  int* sRows = reinterpret_cast<int*>(sth + 32);               // kBack3 * max_col
  // staged schedule tables of two panels (even / odd target panel): owner records, panel record, steps.  Everything the
  // phases look up comes from here -- a phase that chases a dozen dependent L2 loads per warp costs more than its arithmetic
  constexpr int kOwnWords = (int)(sizeof(V3Own) / 4), kPanWords = (int)(sizeof(V3Panel) / 4);
  const int meta_words = kV3Warps * kOwnWords + kPanWords + 4 * P.max_steps;
  int* sMeta = sRows + ((kBack3 * P.max_col + 3) & ~3);        // 2 * meta_words, 16-byte aligned
  __shared__ int s_info;
  __shared__ __align__(8) unsigned long long s_bar[kBack3];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  double* L = work + (int64_t)blockIdx.x * P.work_stride;
  double* zero_tile = win + P.n_win * 64;
  double* acc_rhs = accbuf + 2 * P.acc_rows * 64;
#ifdef LRBMS_DEVTOOLS
  const bool timing = P.timing != nullptr && blockIdx.x == 0;
  long long tph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = 0;
// (the volatile shared-memory read makes a deferred-blocking barrier in front of the tick complete before the clock is read)
#define V3_TICK(k) do { if (timing) { const int dummy_ = *(volatile int*)&s_info; const long long now_ = clock64() + (dummy_ & 0); tph[k] += now_ - tlast; tlast = now_; } } while (0)
#else
#define V3_TICK(k) do { } while (0)
#endif

  // copies the tables of target panel q into its staging buffer (asynchronous; the caller waits and synchronises)
  auto stage_meta = [&](int q, int tid, int nthreads) {
    if (q > P.np) return;
    int* dst = sMeta + (q & 1) * meta_words;
    const int4* osrc = reinterpret_cast<const int4*>(P.own + (size_t)q * kV3Warps);
    for (int i = tid; i < kV3Warps * kOwnWords / 4; i += nthreads) cp_async16(dst + 4 * i, osrc + i);
    if (q < P.np) {
      const int4* psrc = reinterpret_cast<const int4*>(P.pan + q);
      for (int i = tid; i < kPanWords / 4; i += nthreads) cp_async16(dst + kV3Warps * kOwnWords + 4 * i, psrc + i);
      const int st0 = __ldg(&P.pan[q].step0), stn = __ldg(&P.pan[q].n_steps);
      for (int i = tid; i < stn; i += nthreads) cp_async16(dst + kV3Warps * kOwnWords + kPanWords + 4 * i, P.steps + st0 + i);
    }
  };

  for (int64_t mu = blockIdx.x; mu < n_mu; mu += gridDim.x) {
    __syncthreads();
    stage_meta(0, threadIdx.x, kThreads3);
    cp_async_commit();
    for (int q = threadIdx.x; q < P.n_theta; q += kThreads3) sth[q] = theta[mu * P.n_theta + q];
    for (int i = threadIdx.x; i < 64; i += kThreads3) zero_tile[i] = 0.0;
    if (threadIdx.x == 0) s_info = 0;
    cp_async_wait<0>();
    __syncthreads();
#ifdef LRBMS_DEVTOOLS
    if (timing) tlast = clock64();
#endif

    for (int p = -1; p < P.np; ++p) {
      const int q = p + 1;
      const int* metaq = sMeta + (q & 1) * meta_words;
      const V3Own* o = reinterpret_cast<const V3Own*>(metaq) + warp;
      const V3Panel* pq = reinterpret_cast<const V3Panel*>(metaq + kV3Warps * kOwnWords);
      const int4* stq = reinterpret_cast<const int4*>(metaq + kV3Warps * kOwnWords + kPanWords);
      const double* sWp = sW + (p & 1) * 192;                  // diagonal block of panel p (p >= 0)
      double2 acc[2][2];                                       // this warp's own block of panel q (accumulator layout)
      double2 fr[2][2];                                        // its rows of panel p, solved, as fragments [row][column]
      bool own_block = false, is_rhs = false;
      int n_chunks = 0;
      if (warp > 0) {
        n_chunks = o->n_chunks;
        if (n_chunks > 0) {
          own_block = o->chunk_dest[0] == -1;
          is_rhs = o->row[0] == -2;
        }
      }
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int c = 0; c < 2; ++c) { acc[r][c] = make_double2(0.0, 0.0); fr[r][c] = make_double2(0.0, 0.0); }

      // ------------------------------------------------------------------ phase A: early updates of panel q
      if (warp == 0 && q < P.np) {
        // warp 0 has just finished the chain of panel p and waits for the others: bring the operator tiles of the next diagonal
        // block into L1 meanwhile (six dependent L2 / DRAM round trips in front of the next chain otherwise: 4.6 k cycles)
        const int adp[3] = {pq->a_d00, pq->a_d10, pq->a_d11};
#pragma unroll
        for (int k = 0; k < 3; ++k)
          if (adp[k] >= 0)
            for (int qq = 0; qq < P.Q; ++qq)
              asm volatile("prefetch.global.L1 [%0];\n" ::"l"(P.a_tiles + ((int64_t)qq * P.n_a_tiles + adp[k]) * 64 + g * 8 + 2 * t));
      }
      if (warp > 0 && q < P.np) {
        for (int k = 0; k < n_chunks; ++k) {
          const int dest = o->chunk_dest[k];
          if (dest == -2) continue;
          const int kind = o->chunk_kind[k], s0 = o->chunk_step[k], n = o->chunk_n[k];
          double2 a[2][2];
#pragma unroll
          for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int c = 0; c < 2; ++c) a[r][c] = make_double2(0.0, 0.0);
          if (dest == -1 && !is_rhs) {
            // the operator tiles of the block are needed at the END (added to the accumulated updates): start them on their
            // way into L1 now, so that neither the loads nor their latency sit in front of the DMMA chains
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
              for (int c = 0; c < 2; ++c) {
                const int ai = o->amap[r][c];
                if (ai >= 0)
                  for (int qq = 0; qq < P.Q; ++qq)
                    asm volatile("prefetch.global.L1 [%0];\n" ::"l"(P.a_tiles + ((int64_t)qq * P.n_a_tiles + ai) * 64 + g * 8 + 2 * t));
              }
          }
          const int4* stc = stq + (s0 - pq->step0);
#pragma unroll 2
          for (int j = 0; j < n; ++j) {
            const int4 st = stc[j];                            // one broadcast shared-memory load per step
            const double2 fb0 = *reinterpret_cast<const double2*>(win + st.z * 64 + lane * 2);
            const double2 fb1 = *reinterpret_cast<const double2*>(win + st.w * 64 + lane * 2);
            if (kind == 0) {
              const double2 fa0 = *reinterpret_cast<const double2*>(win + st.x * 64 + lane * 2);
              const double2 fa1 = *reinterpret_cast<const double2*>(win + st.y * 64 + lane * 2);
              tile_msub(a[0][0], fa0, fb0);
              tile_msub(a[0][1], fa0, fb1);
              tile_msub(a[1][0], fa1, fb0);
              tile_msub(a[1][1], fa1, fb1);
            } else {
              // forward-substitution row: the A operand is y_K in row 0 of a virtual tile
              const double2 fy = make_double2((g == 0) ? sx[8 * st.x + t] : 0.0, (g == 0) ? sx[8 * st.x + 4 + t] : 0.0);
              tile_msub(a[0][0], fy, fb0);
              tile_msub(a[0][1], fy, fb1);
            }
          }
          if (dest == -1) {
            // + the assembled operator: sum_q theta_q A_q, left to right (LincombOperator.assemble)
            if (is_rhs) {
              if (g == 0) {
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                  double2 f = make_double2(0.0, 0.0);
                  for (int qq = 0; qq < P.Qf; ++qq) {
                    const double2 v = __ldg(reinterpret_cast<const double2*>(P.rhs + (int64_t)qq * P.n_pad + 8 * (2 * q + c) + 2 * t));
                    const double th = sth[P.Q + qq];
                    if (qq == 0) { f.x = th * v.x; f.y = th * v.y; }
                    else { f.x += th * v.x; f.y += th * v.y; }
                  }
                  a[0][c].x += f.x; a[0][c].y += f.y;
                }
              }
            } else {
#pragma unroll
              for (int r = 0; r < 2; ++r)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                  const int ai = o->amap[r][c];
                  if (ai >= 0) {
                    const double* at = P.a_tiles + (int64_t)ai * 64 + g * 8 + 2 * t;
                    double2 f = make_double2(0.0, 0.0);
                    for (int qq = 0; qq < P.Q; ++qq) {
                      const double2 v = __ldg(reinterpret_cast<const double2*>(at + (int64_t)qq * P.n_a_tiles * 64));
                      if (qq == 0) { f.x = sth[0] * v.x; f.y = sth[0] * v.y; }
                      else { f.x += sth[qq] * v.x; f.y += sth[qq] * v.y; }
                    }
                    a[r][c].x += f.x; a[r][c].y += f.y;
                  }
                }
            }
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
              for (int c = 0; c < 2; ++c) acc[r][c] = a[r][c];
          } else {
            double* pb = part + dest * 256 + g * 8 + 2 * t;
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
              for (int c = 0; c < 2; ++c) *reinterpret_cast<double2*>(pb + (r * 2 + c) * 64) = a[r][c];
          }
        }
      }
      V3_TICK(0);
      bar_sync_named(0, kThreads3);        // (as volatile asm: keeps its order with the cycle counters of developer builds)
      V3_TICK(1);
      // the tables of panel q + 1 go into the other staging buffer (its last readers finished before the barrier above)
      if (warp > 0) stage_meta(q + 1, (int)threadIdx.x - 32, kThreads3 - 32);
      cp_async_commit();
      if (warp > 0) V3_TICK(2);

      // ------------------------------------------------------------------ phase B1: solves of panel p
      double2 dd[3];                                           // warp 0: D00, D10, D11 of panel q (accumulator layout)
      double2 hf[2][2];                                        // warp 0: head rows as fragments [row][column of panel p]
      if (warp > 0) {
        if (p >= 0 && own_block) {
          if (is_rhs) {
            double2 x0, x1;
            solve_row(acc_rhs, acc_rhs + 64, sWp, g, t, fr[0][0], fr[0][1], x0, x1);
            if (g == 0) {
              *reinterpret_cast<double2*>(sx + 16 * p + 2 * t) = x0;
              *reinterpret_cast<double2*>(sx + 16 * p + 8 + 2 * t) = x1;
            }
          } else {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
              if (o->row[r] >= 0 && o->prev[r]) {
                double* ct = accbuf + o->acc[r] * 128;
                double2 x0, x1;
                solve_row(ct, ct + 64, sWp, g, t, fr[r][0], fr[r][1], x0, x1);
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                  *reinterpret_cast<double2*>(win + o->wprev[r][c] * 64 + lane * 2) = fr[r][c];
                  *reinterpret_cast<double2*>(L + (int64_t)o->gprev[r][c] * 64 + lane * 2) = fr[r][c];
                }
              }
            }
          }
        }
      } else if (q < P.np) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          hf[r][0] = hf[r][1] = make_double2(0.0, 0.0);
          if (p >= 0 && pq->head_exists[r]) {
            double* ct = accbuf + pq->head_acc[r] * 128;
            double2 x0, x1;
            solve_row(ct, ct + 64, sWp, g, t, hf[r][0], hf[r][1], x0, x1);
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              *reinterpret_cast<double2*>(win + pq->head_w[r][c] * 64 + lane * 2) = hf[r][c];
              *reinterpret_cast<double2*>(L + (int64_t)pq->head_g[r][c] * 64 + lane * 2) = hf[r][c];
            }
          }
        }
        V3_TICK(2);
        // the diagonal block of panel q: operator tiles + the partial blocks of its early updates
        const int ad[3] = {pq->a_d00, pq->a_d10, pq->a_d11};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          dd[k] = make_double2(0.0, 0.0);
          if (ad[k] >= 0) {
            const double* at = P.a_tiles + (int64_t)ad[k] * 64 + g * 8 + 2 * t;
            for (int qq = 0; qq < P.Q; ++qq) {
              const double2 v = __ldg(reinterpret_cast<const double2*>(at + (int64_t)qq * P.n_a_tiles * 64));
              if (qq == 0) { dd[k].x = sth[0] * v.x; dd[k].y = sth[0] * v.y; }
              else { dd[k].x += sth[qq] * v.x; dd[k].y += sth[qq] * v.y; }
            }
          }
        }
#pragma unroll
        for (int k = 0; k < kV3MaxFold; ++k) {
          const int e = pq->fold[k];
          if (e >= 0) {
            const double* pb = part + e * 256 + g * 8 + 2 * t;
            const double2 v00 = *reinterpret_cast<const double2*>(pb), v10 = *reinterpret_cast<const double2*>(pb + 128);
            const double2 v11 = *reinterpret_cast<const double2*>(pb + 192);
            dd[0].x += v00.x; dd[0].y += v00.y; dd[1].x += v10.x; dd[1].y += v10.y; dd[2].x += v11.x; dd[2].y += v11.y;
          }
        }
      }
      // barrier X: the head rows are in the window, warp 0 has read its partial blocks; warp 0 does not wait
      V3_TICK(3);
      if (warp == 0) { __threadfence_block(); bar_arrive_named(2, kThreads3); }
      else bar_sync_named(2, kThreads3);
      V3_TICK(4);

      // ------------------------------------------------------------------ phase B2
      if (warp > 0) {
        if (q < P.np && own_block) {
#pragma unroll
          for (int k = 0; k < kV3MaxFold; ++k) {
            const int e = o->fold[k];
            if (e >= 0) {
              const double* pb = part + e * 256 + g * 8 + 2 * t;
#pragma unroll
              for (int r = 0; r < 2; ++r)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                  const double2 v = *reinterpret_cast<const double2*>(pb + (r * 2 + c) * 64);
                  acc[r][c].x += v.x; acc[r][c].y += v.y;
                }
            }
          }
          if (p >= 0) {
            // late update: target (row r, column t_c) -= sum_s X(r, s) H(c, s)^T, H = head rows of panel p
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              if (!pq->head_exists[c]) continue;
#pragma unroll
              for (int s = 0; s < 2; ++s) {
                const double2 hb = *reinterpret_cast<const double2*>(win + pq->head_w[c][s] * 64 + lane * 2);
                tile_msub(acc[0][c], fr[0][s], hb);
                tile_msub(acc[1][c], fr[1][s], hb);
              }
            }
          }
          if (is_rhs) {
            *reinterpret_cast<double2*>(acc_rhs + g * 8 + 2 * t) = acc[0][0];
            *reinterpret_cast<double2*>(acc_rhs + 64 + g * 8 + 2 * t) = acc[0][1];
          } else {
#pragma unroll
            for (int r = 0; r < 2; ++r)
              if (o->row[r] >= 0) {
                double* ct = accbuf + o->acc[r] * 128 + g * 8 + 2 * t;
                *reinterpret_cast<double2*>(ct) = acc[r][0];
                *reinterpret_cast<double2*>(ct + 64) = acc[r][1];
              }
          }
        }
        V3_TICK(5);
        cp_async_wait<0>();                                    // this thread's share of the next panel's tables has landed
        bar_sync_named(1, kThreads3 - 32);
        V3_TICK(6);
      } else if (q < P.np) {
        // late update of the diagonal block with the head rows, then the critical chain of panel q
        if (p >= 0) {
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            tile_msub(dd[0], hf[0][s], hf[0][s]);
            tile_msub(dd[1], hf[1][s], hf[0][s]);
            tile_msub(dd[2], hf[1][s], hf[1][s]);
          }
        }
        double* sWq = sW + (q & 1) * 192;
        double* t00 = accbuf + pq->acc_rows[0] * 128;  // scratch: the accumulator tiles of the two diagonal rows
        double* t10 = accbuf + pq->acc_rows[1] * 128;
        double* t11 = t10 + 64;
        __syncwarp();
        *reinterpret_cast<double2*>(t00 + g * 8 + 2 * t) = dd[0];
        __syncwarp();
        int bad = potrf_inverse(t00, sWq, L + (int64_t)pq->g_d00 * 64, 16 * q, P.n_red, lane);
        // L10 = D10 W00^T
        const double2 f10in = to_fragment(t10, dd[1], g, t);
        const double2 x10 = tile_times_wt(f10in, sWq, g, t);
        __syncwarp();
        *reinterpret_cast<double2*>(sWq + 64 + g * 8 + 2 * t) = x10;   // row-major: the B operand of C1 -= X0 L10^T
        __syncwarp();
        const double2 f10 = make_double2(sWq[64 + g * 8 + t], sWq[64 + g * 8 + t + 4]);
        *reinterpret_cast<double2*>(L + (int64_t)pq->g_d10 * 64 + lane * 2) = f10;
        tile_msub(dd[2], f10, f10);                            // D11 -= L10 L10^T
        __syncwarp();
        *reinterpret_cast<double2*>(t11 + g * 8 + 2 * t) = dd[2];
        __syncwarp();
        const int bad2 = potrf_inverse(t11, sWq + 128, L + (int64_t)pq->g_d11 * 64, 16 * q + 8, P.n_red, lane);
        if (!bad) bad = bad2;
        if (bad && lane == 0 && s_info == 0) s_info = bad;
        V3_TICK(5);
      }
    }

    // ---------------- backward substitution  L^T u = y (as in solve_kernel_v2): the factor streams back through a ring of
    //                  bulk copies (TMA engine), one tile column per stage; warp 0 finishes u_J while the others already form
    //                  the partial sums of column J - 1.
    {
      const int stage = P.back_stage_doubles;
      auto issue = [&](int Jc) {
        if (Jc >= 0) {
          const int4 col = __ldg(P.ccol + Jc);
          const int sidx = (P.ntc - 1 - Jc) % kBack3;
          double* dst = win + sidx * stage;
          const double* src = L + (int64_t)col.x * 64;
          if (threadIdx.x == 32) {
            mbar_expect_tx(&s_bar[sidx], (unsigned)(col.y * 512));
            bulk_copy_g2s(dst, src, (unsigned)(col.y * 512), &s_bar[sidx]);
          }
          const int tid = (int)threadIdx.x - 64;
          if (tid >= 0 && tid < col.y) cp_async4(sRows + sidx * P.max_col + tid, P.row_idx + col.x + tid);
        }
        cp_async_commit();
      };
      auto wait_column = [&](int Jc) {
        if (Jc >= 0) mbar_wait(&s_bar[(P.ntc - 1 - Jc) % kBack3], (unsigned)(((P.ntc - 1 - Jc) / kBack3) & 1));
      };
      fence_proxy_async_all();                          // the factor was written with st.global; bulk copies read it back
      __syncthreads();
      if (threadIdx.x == 0)
        for (int i = 0; i < kBack3; ++i) mbar_init(&s_bar[i], 1);
      fence_proxy_async();
      for (int i = threadIdx.x; i < 2 * kV3Warps * 8; i += kThreads3) sred[i] = 0.0;
      __syncthreads();
      for (int s = 0; s < kBack3 - 2; ++s) issue(P.ntc - 1 - s);
      cp_async_wait<kBack3 - 4>();
      __syncthreads();
      for (int J = P.ntc - 1; J >= 0; --J) {
        issue(J - (kBack3 - 2));
        if (warp == 0) {
          wait_column(J);
          const int bsel = (P.ntc - 1 - J) % kBack3;
          const double* buf = win + bsel * stage;
          const double* red = sred + (J & 1) * kV3Warps * 8;
          const int cidx = lane & 7, q4 = lane >> 3;
          const double* rq = red + (q4 * 4) * 8 + cidx;
          double partv = (rq[0] + rq[8]) + (rq[16] + rq[24]);
          partv += __shfl_xor_sync(0xffffffffu, partv, 8);
          partv += __shfl_xor_sync(0xffffffffu, partv, 16);
          if (__ldg(P.ccol + J).w) {                     // tile (J + 1, J): the only contribution that needs u_{J+1}
            const double2 f = *reinterpret_cast<const double2*>(buf + 64 + lane * 2);
            const double xv = sx[8 * (J + 1) + g];
            double s0 = f.x * xv, s1 = f.y * xv;
#pragma unroll
            for (int ofs = 4; ofs < 32; ofs <<= 1) {
              s0 += __shfl_xor_sync(0xffffffffu, s0, ofs);
              s1 += __shfl_xor_sync(0xffffffffu, s1, ofs);
            }
            const double v0 = __shfl_sync(0xffffffffu, s0, cidx & 3), v1 = __shfl_sync(0xffffffffu, s1, cidx & 3);
            partv += (cidx < 4) ? v0 : v1;
          }
          const double v = sx[8 * J + cidx] - partv;
          double accv = buf[(2 * q4) * 8 + cidx] * __shfl_sync(0xffffffffu, v, 2 * q4) +
                        buf[(2 * q4 + 1) * 8 + cidx] * __shfl_sync(0xffffffffu, v, 2 * q4 + 1);
          accv += __shfl_xor_sync(0xffffffffu, accv, 8);
          accv += __shfl_xor_sync(0xffffffffu, accv, 16);
          if (lane < 8) sx[8 * J + cidx] = accv;
        } else {
          double s0 = 0.0, s1 = 0.0;
          if (J >= 1) {
            wait_column(J - 1);
            const int bsel = (P.ntc - J) % kBack3;
            const double* buf = win + bsel * stage;
            const int* rws = sRows + bsel * P.max_col;
            const int4 col = __ldg(P.ccol + J - 1);
            for (int li = 1 + col.w + (warp - 1); li < col.y; li += kV3Warps - 1) {
              const double2 f = *reinterpret_cast<const double2*>(buf + li * 64 + lane * 2);
              const double xv = sx[8 * rws[li] + g];
              s0 += f.x * xv;
              s1 += f.y * xv;
            }
#pragma unroll
            for (int ofs = 4; ofs < 32; ofs <<= 1) {
              s0 += __shfl_xor_sync(0xffffffffu, s0, ofs);
              s1 += __shfl_xor_sync(0xffffffffu, s1, ofs);
            }
          }
          double* red = sred + ((J + 1) & 1) * kV3Warps * 8;
          if (g == 0) { red[warp * 8 + t] = s0; red[warp * 8 + 4 + t] = s1; }
        }
        cp_async_wait<kBack3 - 4>();
        __syncthreads();
      }
      cp_async_wait<0>();
    }
    for (int i = threadIdx.x; i < P.n_red; i += kThreads3) u[mu * P.n_red + i] = sx[i];
    if (threadIdx.x == 0 && info) info[mu] = s_info;
    V3_TICK(7);
  }
#ifdef LRBMS_DEVTOOLS
  if (timing && lane == 0)
    for (int k = 0; k < 8; ++k) P.timing[warp * 8 + k] = tph[k];
#endif
#undef V3_TICK
}

}  // namespace

size_t lrbms_v3_smem_bytes(const V3Params& P) {
  return sizeof(double) * ((size_t)P.region_doubles + (size_t)(2 * P.acc_rows + 2) * 64 + (size_t)P.n_partial * 256 + P.n_pad +
                           2 * 3 * 64 + 2 * kV3Warps * 8 + 32) +
         sizeof(int) * ((size_t)((kBack3 * P.max_col + 3) & ~3) + 2 * (size_t)(kV3Warps * (sizeof(V3Own) / 4) + sizeof(V3Panel) / 4 + 4 * (size_t)P.max_steps)) + 16;
}

int lrbms_v3_prepare(lrbms_context* ctx, const V3Params& P, size_t* smem_out) {
  const size_t bytes = lrbms_v3_smem_bytes(P);
  size_t static_bytes = 0;
  cudaError_t e = lrbms_open_dynamic_smem(ctx, (const void*)solve_kernel_v3, &static_bytes);
  if (e != cudaSuccess) return lrbms_fail(ctx, LRBMS_ERR_CUDA, cudaGetErrorString(e));
  if (bytes + static_bytes > (size_t)ctx->max_smem_optin) return LRBMS_ERR_UNSUPPORTED;      // caller falls back
  *smem_out = bytes;
  return LRBMS_OK;
}

void lrbms_v3_launch(const V3Params& P, int grid, size_t smem, int64_t n_mu, const double* theta, double* u, int32_t* info,
                     double* work, cudaStream_t s) {
  solve_kernel_v3<<<grid, kThreads3, smem, s>>>(P, n_mu, theta, u, info, work);
}

int lrbms_v3_back_stages() { return kBack3; }
