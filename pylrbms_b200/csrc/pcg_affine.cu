// Fine-scale solve of an affine operator for a batch of parameters (d.solve(mu) / d.solve_batch(mus)).
//
// The reference assembles A(mu) = sum_q theta_q(mu) A_q and calls apply_inverse once per parameter (dune-istl).  Here the
// Q components live on ONE CSR pattern (values [Q][nnz]) and one Jacobi-preconditioned CG runs for the whole batch: a warp
// takes one matrix row for 32 parameters, lane k = parameter k of the group, so the row's column indices and Q value arrays
// are read once per group (warp-uniform loads) and the vectors x[c][32 g : 32 g + 32] with one coalesced 256-byte access.
// Every lane forms sum_q theta_q v_q in registers.  Vectors are dof-major [n][m_pad], m_pad = n_mu rounded up to 32.
//
// Bits of one parameter do not depend on the batch: a row sum runs sequentially in CSR order inside one lane; an inner
// product adds, per parameter, the rows of a warp in order, the 32 warps of a CTA in order and the CTAs in order, over a
// row partition fixed by n and the SM count only.  Nothing a lane computes reads another parameter's numbers.  Parameters
// are stopped, restarted and frozen on their own at fixed check points (every kCheck iterations) by the host, from their
// own scalars only; a frozen parameter gets alpha = 0 and none of its columns is written again.
//
// One cooperative launch runs kCheck iterations (two grid-wide barriers per iteration, as pcg_iterate_kernel); there is
// no multi-launch variant, which would sum in a different order.
#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int kThreads = 1024;
constexpr int kWarps = kThreads / 32;
constexpr int kCheck = 25;
constexpr int kMaxQ = 4;
constexpr int kPadLane = 3;   // status of the padding lanes n_mu <= m < m_pad

// status: -1 active, 0 converged, 1 not converged, 2 p^T A p <= 0, kPadLane padding
struct AffVecs {
  double *r, *z, *p0, *p1, *Ap, *dinv;         // [n][m_pad]
  double *part_a, *part_b, *part_c;            // [grid][m_pad]
  double *rz, *rz_prev, *rr, *bb;              // [m_pad]
  int *status, *cmd, *iters, *k_local;         // [m_pad]; cmd != 0: recompute the true residual (restart)
};

inline int aff_grid(const lrbms_context* ctx, int64_t n) {
  return (int)std::max<int64_t>(1, std::min<int64_t>(ctx->sm_count, (n + kWarps - 1) / kWarps));
}

inline int64_t aff_m_pad(int64_t n_mu) { return (n_mu + 31) / 32 * 32; }

inline size_t aff_ws_bytes(int64_t n, int64_t m_pad, int grid) {
  return sizeof(double) * ((size_t)6 * n * m_pad + (size_t)3 * grid * m_pad + (size_t)4 * m_pad) + sizeof(int) * 4 * (size_t)m_pad;
}

inline size_t aff_smem_bytes(int64_t m_pad) { return sizeof(double) * (32 * 32 + 3 * (size_t)m_pad) + sizeof(int) * 3 * (size_t)m_pad; }

__device__ __forceinline__ void cta_rows(int n, int* r0, int* r1) {
  *r0 = (int)((int64_t)n * blockIdx.x / gridDim.x);
  *r1 = (int)((int64_t)n * (blockIdx.x + 1) / gridDim.x);
}

// per-parameter CTA partial: the 32 warps' sums added in warp order; red: 32 x 32 doubles
__device__ __forceinline__ void cta_partial(double v, double* red, double* part, int m) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  red[warp * 32 + lane] = v;
  __syncthreads();
  if (warp == 0) {
    double s = 0.0;
    for (int w = 0; w < kWarps; ++w) s += red[w * 32 + lane];
    __stcg(part + m, s);
  }
  __syncthreads();
}

// the same value in every CTA: the CTA partials of parameter m added in CTA order
__device__ __forceinline__ double all_ctas(const double* part, int n_part, int64_t m_pad, int m) {
  double s = 0.0;
  for (int c = 0; c < n_part; ++c) s += __ldcg(part + c * m_pad + m);
  return s;
}

template <int Q>
__device__ __forceinline__ double coef(const double (&th)[Q], const double* __restrict__ values, int64_t nnz, int k) {
  double a = th[0] * __ldg(values + k);
#pragma unroll
  for (int q = 1; q < Q; ++q) a = fma(th[q], __ldg(values + q * nnz + k), a);
  return a;
}

// Restart of the parameters with cmd != 0: b = sum_f theta_f rhs_f, r = b - A x, dinv = 1 / diag(A), z = dinv r; CTA
// partials of b.b (part_a), r.z (part_b), r.r (part_c).  Same grid and row partition as the iteration kernel.
template <int Q>
__global__ void __launch_bounds__(kThreads, 1) affine_restart_kernel(int n, const int32_t* __restrict__ rowptr,
                                                                     const int32_t* __restrict__ colind,
                                                                     const double* __restrict__ values, int64_t nnz, int Qf,
                                                                     const double* __restrict__ rhs,
                                                                     const double* __restrict__ theta, int64_t m_pad,
                                                                     const double* __restrict__ x, int ldx, AffVecs V) {
  __shared__ double red[32 * 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int r0, r1;
  cta_rows(n, &r0, &r1);
  for (int g = 0; g < (int)(m_pad / 32); ++g) {
    const int m = g * 32 + lane;
    const bool on = V.cmd[m] != 0;
    if (!__any_sync(0xffffffffu, on)) continue;            // the same in every warp: V.cmd is not written here
    double th[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) th[q] = on ? theta[(int64_t)m * (Q + Qf) + q] : 0.0;
    double bb = 0.0, rz = 0.0, rr = 0.0;
    for (int row = r0 + warp; row < r1; row += kWarps) {
      double ax = 0.0, d = 0.0;
      const int k1 = __ldg(rowptr + row + 1);
      for (int k = __ldg(rowptr + row); k < k1; ++k) {
        const int c = __ldg(colind + k);
        const double a = coef<Q>(th, values, nnz, k);
        if (on) ax = fma(a, x[(int64_t)c * ldx + m], ax);
        if (c == row) d = a;
      }
      if (on) {
        double b = 0.0;
        for (int f = 0; f < Qf; ++f) b = fma(theta[(int64_t)m * (Q + Qf) + Q + f], __ldg(rhs + (int64_t)f * n + row), b);
        const double rv = b - ax, di = (d != 0.0) ? 1.0 / d : 1.0, zv = di * rv;
        const int64_t o = (int64_t)row * m_pad + m;
        __stcg(V.r + o, rv); __stcg(V.z + o, zv); __stcg(V.dinv + o, di);
        bb = fma(b, b, bb); rz = fma(rv, zv, rz); rr = fma(rv, rv, rr);
      }
    }
    const int64_t po = (int64_t)blockIdx.x * m_pad + g * 32;
    cta_partial(bb, red, V.part_a + po, lane);
    cta_partial(rz, red, V.part_b + po, lane);
    cta_partial(rr, red, V.part_c + po, lane);
  }
}

__global__ void affine_restart_scalars_kernel(int n_part, int64_t m_pad, AffVecs V) {
  for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < m_pad; m += gridDim.x * blockDim.x) {
    if (V.cmd[m] == 0) continue;
    V.bb[m] = all_ctas(V.part_a, n_part, m_pad, m);
    V.rz[m] = all_ctas(V.part_b, n_part, m_pad, m);
    V.rr[m] = all_ctas(V.part_c, n_part, m_pad, m);
    V.rz_prev[m] = 0.0;
    V.k_local[m] = 0;
  }
}

// n_it CG iterations for every active parameter.  Per-parameter scalars sit in shared memory, derived identically in
// every CTA; CTA 0 publishes them at the end.  The direction update p = z + beta p is folded into the product as in
// pcg_iterate_kernel: every lane forms the entries of the new p it reads (the same fma as the row's owner, so the same
// bits), the owner stores them into the other p buffer.
template <int Q>
__global__ void __launch_bounds__(kThreads, 1) affine_iterate_kernel(int n, const int32_t* __restrict__ rowptr,
                                                                     const int32_t* __restrict__ colind,
                                                                     const double* __restrict__ values, int64_t nnz,
                                                                     const double* __restrict__ theta, int ldt, int64_t m_pad,
                                                                     double* x, int ldx, AffVecs V, int it0, int n_it) {
  cg::grid_group grid = cg::this_grid();
  extern __shared__ double smem[];
  double* red = smem;
  double* s_rz = red + 32 * 32;
  double* s_rzp = s_rz + m_pad;
  double* s_coef = s_rzp + m_pad;                          // beta in the product phase, alpha in the update phase
  int* s_st = (int*)(s_coef + m_pad);
  int* s_k = s_st + m_pad;
  int* s_it = s_k + m_pad;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_groups = (int)(m_pad / 32);
  for (int m = threadIdx.x; m < m_pad; m += kThreads) {
    s_rz[m] = __ldcg(V.rz + m); s_rzp[m] = __ldcg(V.rz_prev + m);
    s_st[m] = __ldcg(V.status + m); s_k[m] = __ldcg(V.k_local + m); s_it[m] = __ldcg(V.iters + m);
  }
  __syncthreads();
  int r0, r1;
  cta_rows(n, &r0, &r1);
  for (int kk = 0; kk < n_it; ++kk) {
    const int it = it0 + kk;
    const double* p_old = (it & 1) ? V.p1 : V.p0;
    double* p_new = (it & 1) ? V.p0 : V.p1;
    for (int m = threadIdx.x; m < m_pad; m += kThreads) s_coef[m] = (s_k[m] == 0 || s_rzp[m] == 0.0) ? 0.0 : s_rz[m] / s_rzp[m];
    __syncthreads();
    // ---- p_new = z + beta p_old (own rows stored);  Ap = A(mu) p_new;  partials of p_new.Ap
    for (int g = 0; g < n_groups; ++g) {
      const int m = g * 32 + lane;
      const bool act = s_st[m] < 0;
      if (!__any_sync(0xffffffffu, act)) continue;        // uniform over the CTA: s_st is not written in this phase
      const bool fresh = s_k[m] == 0;                      // first iteration after a (re)start: p = z
      const double beta = s_coef[m];
      double th[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) th[q] = act ? theta[(int64_t)m * ldt + q] : 0.0;
      double pap = 0.0;
      for (int row = r0 + warp; row < r1; row += kWarps) {
        double s = 0.0;
        const int k1 = __ldg(rowptr + row + 1);
        for (int k = __ldg(rowptr + row); k < k1; k += 4) {
          // the loads of four entries are issued before their fmas (latency), which still add in CSR order
          double a[4], v[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const bool in = k + j < k1;
            const int64_t o = (int64_t)(in ? __ldg(colind + k + j) : 0) * m_pad + m;
            a[j] = in ? coef<Q>(th, values, nnz, k + j) : 0.0;
            v[j] = 0.0;
            if (in && act) {
              const double zc = __ldcg(V.z + o);
              v[j] = fresh ? zc : fma(beta, __ldcg(p_old + o), zc);
            }
          }
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (k + j < k1) s = fma(a[j], v[j], s);
        }
        if (act) {
          const int64_t o = (int64_t)row * m_pad + m;
          const double zr = __ldcg(V.z + o);
          const double pv = fresh ? zr : fma(beta, __ldcg(p_old + o), zr);
          __stcg(p_new + o, pv);
          __stcg(V.Ap + o, s);
          pap = fma(pv, s, pap);
        }
      }
      cta_partial(pap, red, V.part_a + (int64_t)blockIdx.x * m_pad + g * 32, lane);
    }
    grid.sync();
    // ---- alpha = rz / p.Ap (p.Ap <= 0 with rz != 0: freeze with status 2);  x += alpha p;  r -= alpha Ap;  z = dinv r
    for (int m = threadIdx.x; m < m_pad; m += kThreads) {
      double alpha = 0.0;
      if (s_st[m] < 0) {
        const double pap = all_ctas(V.part_a, gridDim.x, m_pad, m);
        if (pap > 0.0) alpha = s_rz[m] / pap;
        else if (s_rz[m] != 0.0) s_st[m] = 2;
      }
      s_coef[m] = alpha;
    }
    __syncthreads();
    for (int g = 0; g < n_groups; ++g) {
      const int m = g * 32 + lane;
      const bool act = s_st[m] < 0;
      if (!__any_sync(0xffffffffu, act)) continue;
      const double alpha = s_coef[m];
      double rz = 0.0, rr = 0.0;
      if (act) {
        for (int row = r0 + warp; row < r1; row += kWarps) {
          const int64_t o = (int64_t)row * m_pad + m;
          double* xp = x + (int64_t)row * ldx + m;
          *xp = fma(alpha, __ldcg(p_new + o), *xp);
          const double rv = fma(-alpha, __ldcg(V.Ap + o), __ldcg(V.r + o));
          const double zv = __ldcg(V.dinv + o) * rv;
          __stcg(V.r + o, rv);
          __stcg(V.z + o, zv);
          rz = fma(rv, zv, rz); rr = fma(rv, rv, rr);
        }
      }
      const int64_t po = (int64_t)blockIdx.x * m_pad + g * 32;
      cta_partial(rz, red, V.part_b + po, lane);
      cta_partial(rr, red, V.part_c + po, lane);
    }
    grid.sync();
    for (int m = threadIdx.x; m < m_pad; m += kThreads) {
      if (s_st[m] < 0) {
        s_rzp[m] = s_rz[m];
        s_rz[m] = all_ctas(V.part_b, gridDim.x, m_pad, m);
        s_k[m] += 1;
        s_it[m] += 1;
      }
    }
    __syncthreads();
  }
  if (blockIdx.x == 0) {
    for (int m = threadIdx.x; m < m_pad; m += kThreads) {
      if (s_st[m] < 0 && n_it > 0) __stcg(V.rr + m, all_ctas(V.part_c, gridDim.x, m_pad, m));
      __stcg(V.rz + m, s_rz[m]); __stcg(V.rz_prev + m, s_rzp[m]);
      __stcg(V.status + m, s_st[m]); __stcg(V.k_local + m, s_k[m]); __stcg(V.iters + m, s_it[m]);
    }
  }
}

struct Kernels {
  const void* restart;
  const void* iterate;
};

template <int Q>
Kernels kernels_for() {
  return {(const void*)affine_restart_kernel<Q>, (const void*)affine_iterate_kernel<Q>};
}

inline Kernels kernels_for_q(int Q) {
  switch (Q) {
    case 1: return kernels_for<1>();
    case 2: return kernels_for<2>();
    case 3: return kernels_for<3>();
    default: return kernels_for<4>();
  }
}

inline double rel_res(double rr, double bb) { return (bb > 0.0) ? std::sqrt(rr / bb) : std::sqrt(rr); }

}  // namespace

extern "C" {

int lrbms_affine_pcg_workspace_bytes(lrbms_handle_t h, int64_t n, int64_t n_mu, size_t* bytes) {
  LRBMS_REQUIRE(h, h && bytes && n >= 0 && n_mu >= 0, "affine_pcg_workspace_bytes: bad argument");
  *bytes = aff_ws_bytes(n, aff_m_pad(n_mu), aff_grid(h, n));
  return LRBMS_OK;
}

int lrbms_affine_pcg_solve(lrbms_handle_t h, int32_t n, int32_t Q, const int32_t* rowptr, const int32_t* colind,
                           const double* values, int32_t Qf, const double* rhs, int64_t n_mu, const double* theta,
                           double* x, int32_t ldx, double rtol, int32_t max_iter, int32_t max_restarts,
                           int32_t* iters_out, double* relres_out, int32_t* status_out,
                           void* workspace, size_t workspace_bytes, void* stream) {
  LRBMS_REQUIRE(h, h && rowptr && colind && values && theta && x && workspace, "affine_pcg_solve: null argument");
  LRBMS_REQUIRE(h, iters_out && relres_out && status_out, "affine_pcg_solve: null output array");
  LRBMS_REQUIRE(h, n >= 0 && n_mu >= 0 && Q >= 1 && Qf >= 0 && (Qf == 0 || rhs) && ldx >= n_mu && max_iter >= 0 &&
                       max_restarts >= 0 && rtol >= 0.0, "affine_pcg_solve: bad argument");
  if (Q > kMaxQ) return lrbms_fail(h, LRBMS_ERR_UNSUPPORTED, "affine_pcg_solve: at most 4 affine operator terms are supported");
  const int64_t m_pad = aff_m_pad(n_mu);
  const int grid = aff_grid(h, n);
  LRBMS_REQUIRE(h, workspace_bytes >= aff_ws_bytes(n, m_pad, grid),
                "affine_pcg_solve: workspace too small (see lrbms_affine_pcg_workspace_bytes)");
  for (int64_t m = 0; m < n_mu; ++m) { iters_out[m] = 0; relres_out[m] = 0.0; status_out[m] = 0; }
  if (n == 0 || n_mu == 0) return LRBMS_OK;
  LRBMS_CUDA_CHECK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const Kernels K = kernels_for_q(Q);
  const size_t smem = aff_smem_bytes(m_pad);
  if (smem > (size_t)h->max_smem_optin)
    return lrbms_fail(h, LRBMS_ERR_UNSUPPORTED, "affine_pcg_solve: too many parameters for one call (split the batch)");
  LRBMS_CUDA_CHECK(h, lrbms_open_dynamic_smem(h, K.iterate));
  int coop_attr = 0, per_sm = 0;
  LRBMS_CUDA_CHECK(h, cudaDeviceGetAttribute(&coop_attr, cudaDevAttrCooperativeLaunch, h->device));
  LRBMS_CUDA_CHECK(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, K.iterate, kThreads, smem));
  if (!coop_attr || per_sm < 1)
    return lrbms_fail(h, LRBMS_ERR_UNSUPPORTED, "affine_pcg_solve: the device cannot run the solve kernel as a cooperative "
                                                "launch (one resident CTA of 1024 threads per SM is required)");
  // workspace
  double* w = (double*)workspace;
  const size_t nv = (size_t)n * m_pad;
  AffVecs V;
  V.r = w; V.z = w + nv; V.p0 = w + 2 * nv; V.p1 = w + 3 * nv; V.Ap = w + 4 * nv; V.dinv = w + 5 * nv;
  V.part_a = w + 6 * nv; V.part_b = V.part_a + (size_t)grid * m_pad; V.part_c = V.part_b + (size_t)grid * m_pad;
  V.rz = V.part_c + (size_t)grid * m_pad; V.rz_prev = V.rz + m_pad; V.rr = V.rz_prev + m_pad; V.bb = V.rr + m_pad;
  V.status = (int*)(V.bb + m_pad); V.cmd = V.status + m_pad; V.iters = V.cmd + m_pad; V.k_local = V.iters + m_pad;
  int32_t nnz32 = 0;                                      // values holds Q arrays of rowptr[n] entries
  LRBMS_CUDA_CHECK(h, cudaMemcpyAsync(&nnz32, rowptr + n, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  LRBMS_CUDA_CHECK(h, cudaStreamSynchronize(s));
  int64_t nnz = nnz32, mp = m_pad;
  int ldt = Q + Qf;

  // host copies: status and cmd are uploaded as one block before every launch that reads them
  std::vector<int> ints(3 * m_pad, 0);                    // [status | cmd | iters]
  int* st = ints.data();
  int* cmd = st + m_pad;
  for (int64_t m = 0; m < m_pad; ++m) { st[m] = m < n_mu ? -1 : kPadLane; cmd[m] = m < n_mu ? 1 : 0; }
  std::vector<double> dbl(2 * m_pad);                     // read back: rr, bb
  std::vector<int> dev_st(m_pad);
  std::vector<double> tprev(n_mu, 0.0);
  std::vector<int> n_restart(n_mu, 0);
  std::vector<char> fresh(n_mu, 0);

  auto read_back = [&]() -> int {
    LRBMS_CUDA_CHECK(h, cudaMemcpyAsync(dbl.data(), V.rr, sizeof(double) * 2 * m_pad, cudaMemcpyDeviceToHost, s));
    LRBMS_CUDA_CHECK(h, cudaMemcpyAsync(dev_st.data(), V.status, sizeof(int) * m_pad, cudaMemcpyDeviceToHost, s));
    LRBMS_CUDA_CHECK(h, cudaMemcpyAsync(iters_out, V.iters, sizeof(int) * n_mu, cudaMemcpyDeviceToHost, s));
    LRBMS_CUDA_CHECK(h, cudaStreamSynchronize(s));
    return LRBMS_OK;
  };
  // true residual of every parameter with cmd set; clears cmd on the host
  auto restart = [&](bool first) -> int {
    LRBMS_CUDA_CHECK(h, cudaMemcpyAsync(V.status, ints.data(), sizeof(int) * (first ? 3 : 2) * m_pad, cudaMemcpyHostToDevice, s));
    void* args[] = {(void*)&n, (void*)&rowptr, (void*)&colind, (void*)&values, (void*)&nnz,
                    (void*)&Qf, (void*)&rhs, (void*)&theta, (void*)&mp, (void*)&x, (void*)&ldx,
                    (void*)&V};
    LRBMS_CUDA_CHECK(h, cudaLaunchKernel(K.restart, dim3(grid), dim3(kThreads), args, 0, s));
    affine_restart_scalars_kernel<<<(unsigned)((m_pad + 255) / 256), 256, 0, s>>>(grid, m_pad, V);
    LRBMS_CUDA_CHECK(h, cudaGetLastError());
    int rc = read_back();
    if (rc) return rc;
    for (int64_t m = 0; m < n_mu; ++m)
      if (cmd[m]) { relres_out[m] = rel_res(dbl[m], dbl[m_pad + m]); fresh[m] = 1; cmd[m] = 0; }
    return LRBMS_OK;
  };

  int rc = restart(true);
  if (rc) return rc;
  for (int64_t m = 0; m < n_mu; ++m) {
    tprev[m] = relres_out[m];
    if (relres_out[m] <= rtol) st[m] = 0;
  }
  int it = 0;
  for (;;) {
    bool any = false;
    for (int64_t m = 0; m < n_mu; ++m) any = any || st[m] < 0;
    if (!any) break;
    if (it >= max_iter) {                                  // out of iterations: status 1 with the true residual
      bool need = false;
      for (int64_t m = 0; m < n_mu; ++m)
        if (st[m] < 0) { st[m] = 1; cmd[m] = !fresh[m]; need = need || cmd[m]; }
      if (need && (rc = restart(false))) return rc;
      break;
    }
    int n_it = std::min(kCheck, max_iter - it);
    LRBMS_CUDA_CHECK(h, cudaMemcpyAsync(V.status, st, sizeof(int) * m_pad, cudaMemcpyHostToDevice, s));
    int it0 = it;
    void* args[] = {(void*)&n, (void*)&rowptr, (void*)&colind, (void*)&values, (void*)&nnz,
                    (void*)&theta, (void*)&ldt, (void*)&mp, (void*)&x, (void*)&ldx, (void*)&V,
                    (void*)&it0, (void*)&n_it};
    LRBMS_CUDA_CHECK(h, cudaLaunchCooperativeKernel(K.iterate, dim3(grid), dim3(kThreads), args, smem, s));
    it += n_it;
    if ((rc = read_back())) return rc;
    bool need = false;
    for (int64_t m = 0; m < n_mu; ++m) {
      if (st[m] >= 0) continue;
      fresh[m] = 0;
      if (dev_st[m] == 2) st[m] = 2;                       // frozen by the kernel; report its true residual
      // after a restart the recurrence goes on to 0.1 rtol: its residual runs ahead of the true one (as in the corrector)
      const double target = n_restart[m] ? 0.1 * rtol : rtol;
      if (dev_st[m] == 2 || rel_res(dbl[m], dbl[m_pad + m]) <= target) { cmd[m] = 1; need = true; }
    }
    if (!need) continue;
    std::vector<char> converging(n_mu, 0);
    for (int64_t m = 0; m < n_mu; ++m) converging[m] = cmd[m] && st[m] < 0;
    if ((rc = restart(false))) return rc;
    // the recurrence residual reached rtol: the true one decides (converged / restart while it halves / give up)
    for (int64_t m = 0; m < n_mu; ++m) {
      if (!converging[m]) continue;
      const double t = relres_out[m];
      n_restart[m] += 1;
      if (t <= rtol) st[m] = 0;
      else if (n_restart[m] > max_restarts || !(t < 0.5 * tprev[m])) st[m] = 1;
      else tprev[m] = t;
    }
  }
  for (int64_t m = 0; m < n_mu; ++m) status_out[m] = st[m];
  return LRBMS_OK;
}

}  // extern "C"
