// Reduction error of a parameter batch on the device (reduction_error_analysis): the reconstruction error
// e = u_h - R u_N of every subdomain in one launch, and segmented affine quadratic forms e^T (sum_q theta_q A_q) e per
// row segment (the local energy products, or |||e|||_mu^2 over the whole operator).
//
// Layouts are those of the fine-scale solve (pcg_affine.cu): vectors are dof-major [n][ld], column = parameter, and a warp
// takes one matrix row for 32 parameters, lane = parameter, so a row's column indices, Q value arrays and basis entries
// are warp-uniform loads and the vector entries of 32 parameters one coalesced 256-byte access.
//
// Bits of one parameter do not depend on the batch: e[r][m] is a sequential fma chain over k inside one lane; a form adds,
// per parameter, the rows of a warp in order (each row sum sequential in CSR order), the warps of a CTA in order and the
// CTAs of a segment in order, over a row partition fixed by the segment sizes and the SM count only.  No atomics.
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kCtasPerSm = 8;        // target CTAs per SM of the row partition (latency: each warp walks its rows in turn)
constexpr int kChunk = 256;          // parameters per form launch (shared accumulators [kWarps][kChunk])
constexpr int kMaxQ = 4;

struct CtaRange {
  int32_t seg, r0, r1, pad;          // global rows [r0, r1) of segment seg
};

struct ReconDev {
  const double* V;
  int64_t ldv, row0;
  int32_t N, red_off;
};

// CTAs of every segment: ceil(n_s / R) CTAs with R = max(kWarps, ceil(sum n_s / (kCtasPerSm * sm_count))) rows each at
// most, the rows split evenly; a function of the segment sizes and the SM count only.
void partition(const std::vector<int64_t>& seg_r0, const std::vector<int64_t>& seg_n, int sm_count,
               std::vector<CtaRange>* ctas, std::vector<int32_t>* seg_cta_ptr) {
  int64_t total = 0;
  for (int64_t n_s : seg_n) total += n_s;
  const int64_t target = (int64_t)kCtasPerSm * std::max(1, sm_count);
  const int64_t R = std::max<int64_t>(kWarps, (total + target - 1) / target);
  ctas->clear();
  if (seg_cta_ptr) seg_cta_ptr->assign(1, 0);
  for (size_t s = 0; s < seg_n.size(); ++s) {
    const int64_t n_s = seg_n[s], c_s = (n_s + R - 1) / R;
    for (int64_t j = 0; j < c_s; ++j)
      ctas->push_back({(int32_t)s, (int32_t)(seg_r0[s] + n_s * j / c_s), (int32_t)(seg_r0[s] + n_s * (j + 1) / c_s), 0});
    if (seg_cta_ptr) seg_cta_ptr->push_back((int32_t)ctas->size());
  }
}

inline size_t align256(size_t b) { return (b + 255) / 256 * 256; }

// rows of warp w inside its CTA: a contiguous slice (neighbouring rows share columns, whose entries then come from L1)
__device__ __forceinline__ void warp_rows(const CtaRange& cr, int w, int* w0, int* w1) {
  const int n = cr.r1 - cr.r0;
  *w0 = cr.r0 + (int)((int64_t)n * w / kWarps);
  *w1 = cr.r0 + (int)((int64_t)n * (w + 1) / kWarps);
}

// ---- (a) e[r][m] = u_h[r][m] - sum_{k < N_i} V_i[r - row0_i][k] u_N[m][off_i + k], k ascending.  The coefficients are
// read from the transposed copy c[k][m] (c_t_kernel), so that the 32 lanes of a warp load one 256-byte line per k.
__global__ void c_t_kernel(const double* __restrict__ un, int64_t ldn, int n_mu, int n_red, double* __restrict__ ct,
                           int64_t ldc) {
  const int64_t total = (int64_t)n_red * n_mu;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(i / n_mu), m = (int)(i % n_mu);
    ct[(int64_t)k * ldc + m] = un[(int64_t)m * ldn + k];
  }
}

__global__ void __launch_bounds__(kThreads) recon_error_kernel(const ReconDev* __restrict__ blocks,
                                                               const CtaRange* __restrict__ ctas,
                                                               const double* __restrict__ uh, int64_t ldu,
                                                               const double* __restrict__ ct, int64_t ldc,
                                                               double* __restrict__ e, int64_t lde, int n_mu) {
  const CtaRange cr = ctas[blockIdx.x];
  const ReconDev B = blocks[cr.seg];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_groups = (n_mu + 31) / 32;
  int w0, w1;
  warp_rows(cr, warp, &w0, &w1);
  for (int row = w0; row < w1; ++row) {
    const double* v = B.V + (row - B.row0) * B.ldv;
    for (int g = 0; g < n_groups; ++g) {
      const int m = g * 32 + lane;
      if (m >= n_mu) continue;
      const double* c = ct + (int64_t)B.red_off * ldc + m;
      double s = 0.0;
      for (int k = 0; k < B.N; k += 4) {
        // the loads of four terms are issued before their fmas (latency), which still add in ascending k
        double a[4], b[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const bool in = k + j < B.N;
          a[j] = in ? __ldg(v + k + j) : 0.0;
          b[j] = in ? __ldg(c + (int64_t)(k + j) * ldc) : 0.0;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (k + j < B.N) s = fma(a[j], b[j], s);
      }
      __stcg(e + (int64_t)row * lde + m, __ldg(uh + (int64_t)row * ldu + m) - s);
    }
  }
}

// ---- (b) CTA partials of sum_{r in rows} x[r][m] * sum_c (sum_q theta[m][q] A_q[r][c]) x[c][m] for the parameters
// m0 .. m0 + n_mu_c (n_mu_c <= kChunk); theta == nullptr: theta = 1
template <int Q>
__global__ void __launch_bounds__(kThreads) segmented_form_kernel(const int32_t* __restrict__ rowptr,
                                                                  const int32_t* __restrict__ colind,
                                                                  const double* __restrict__ values, int64_t nnz,
                                                                  const double* __restrict__ theta, int64_t ldt,
                                                                  const double* __restrict__ x, int64_t ldx, int n_mu_c,
                                                                  const CtaRange* __restrict__ ctas, double* __restrict__ part) {
  __shared__ double s_th[Q][kChunk];
  __shared__ double s_acc[kWarps][kChunk];
  const CtaRange cr = ctas[blockIdx.x];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int m = threadIdx.x; m < kChunk; m += kThreads) {
#pragma unroll
    for (int q = 0; q < Q; ++q) s_th[q][m] = (theta && m < n_mu_c) ? theta[(int64_t)m * ldt + q] : 1.0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) s_acc[w][m] = 0.0;
  }
  __syncthreads();
  const int n_groups = (n_mu_c + 31) / 32;
  int w0, w1;
  warp_rows(cr, warp, &w0, &w1);
  for (int row = w0; row < w1; ++row) {
    const int k0 = __ldg(rowptr + row), k1 = __ldg(rowptr + row + 1);
    for (int g = 0; g < n_groups; ++g) {
      const int m = g * 32 + lane;
      const bool act = m < n_mu_c;
      double th[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) th[q] = s_th[q][m];
      double s = 0.0;
      for (int k = k0; k < k1; k += 4) {
        double a[4], v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const bool in = k + j < k1;
          const int c = in ? __ldg(colind + k + j) : 0;
          double aq = 0.0;
          if (in) {
            aq = th[0] * __ldg(values + k + j);
#pragma unroll
            for (int q = 1; q < Q; ++q) aq = fma(th[q], __ldg(values + q * nnz + k + j), aq);
          }
          a[j] = aq;
          v[j] = (in && act) ? __ldg(x + (int64_t)c * ldx + m) : 0.0;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (k + j < k1) s = fma(a[j], v[j], s);
      }
      if (act) s_acc[warp][m] = fma(__ldg(x + (int64_t)row * ldx + m), s, s_acc[warp][m]);
    }
  }
  __syncthreads();
  for (int m = threadIdx.x; m < n_mu_c; m += kThreads) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) t += s_acc[w][m];
    part[(int64_t)blockIdx.x * kChunk + m] = t;
  }
}

// out[s][m] = the CTA partials of segment s added in CTA order (0 for a segment without rows)
__global__ void segment_sum_kernel(const double* __restrict__ part, const int32_t* __restrict__ seg_cta_ptr, int n_seg,
                                   int n_mu_c, double* __restrict__ out, int64_t ldo) {
  const int64_t total = (int64_t)n_seg * n_mu_c;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i / n_mu_c), m = (int)(i % n_mu_c);
    double t = 0.0;
    for (int c = seg_cta_ptr[s]; c < seg_cta_ptr[s + 1]; ++c) t += part[(int64_t)c * kChunk + m];
    out[(int64_t)s * ldo + m] = t;
  }
}

const void* form_kernel_for_q(int Q) {
  switch (Q) {
    case 1: return (const void*)segmented_form_kernel<1>;
    case 2: return (const void*)segmented_form_kernel<2>;
    case 3: return (const void*)segmented_form_kernel<3>;
    default: return (const void*)segmented_form_kernel<4>;
  }
}

void recon_partition(const lrbms_recon_block_t* blocks, int n_sub, int sm_count, std::vector<CtaRange>* ctas) {
  std::vector<int64_t> r0(n_sub), n(n_sub);
  for (int i = 0; i < n_sub; ++i) { r0[i] = blocks[i].row_offset; n[i] = blocks[i].n_rows; }
  partition(r0, n, sm_count, ctas, nullptr);
}

void form_partition(int n_seg, const int32_t* seg_ptr, int sm_count, std::vector<CtaRange>* ctas, std::vector<int32_t>* seg_cta) {
  std::vector<int64_t> r0(n_seg), n(n_seg);
  for (int s = 0; s < n_seg; ++s) { r0[s] = seg_ptr[s]; n[s] = (int64_t)seg_ptr[s + 1] - seg_ptr[s]; }
  partition(r0, n, sm_count, ctas, seg_cta);
}

inline int64_t recon_ldc(int64_t n_mu) { return (n_mu + 31) / 32 * 32; }

inline size_t recon_ws_bytes(int n_sub, size_t n_cta, int64_t n_mu, int64_t n_red) {
  return align256(sizeof(double) * (size_t)n_red * recon_ldc(n_mu)) + align256(sizeof(ReconDev) * (size_t)n_sub) +
         sizeof(CtaRange) * n_cta;
}

inline size_t form_ws_bytes(int n_seg, size_t n_cta) {
  return align256(sizeof(double) * kChunk * n_cta) + align256(sizeof(CtaRange) * n_cta) + sizeof(int32_t) * ((size_t)n_seg + 1);
}

int check_recon_blocks(lrbms_handle_t h, int n_sub, const lrbms_recon_block_t* b) {
  int64_t prev_end = 0;
  for (int i = 0; i < n_sub; ++i) {
    LRBMS_REQUIRE(h, b[i].n_rows >= 0 && b[i].row_offset >= prev_end && b[i].row_offset + b[i].n_rows <= INT32_MAX,
                  "recon_error: block " + std::to_string(i) + ": rows must be ascending, disjoint and below 2^31");
    prev_end = b[i].row_offset + b[i].n_rows;
  }
  return LRBMS_OK;
}

}  // namespace

extern "C" {

int lrbms_recon_error_workspace_bytes(lrbms_handle_t h, int32_t n_sub, const lrbms_recon_block_t* blocks_host, int64_t n_mu,
                                      int32_t n_red, size_t* bytes) {
  LRBMS_REQUIRE(h, h && bytes && n_sub >= 0 && (n_sub == 0 || blocks_host) && n_mu >= 0 && n_red >= 0,
                "recon_error_workspace_bytes: bad argument");
  int rc = check_recon_blocks(h, n_sub, blocks_host);
  if (rc) return rc;
  std::vector<CtaRange> ctas;
  recon_partition(blocks_host, n_sub, h->sm_count, &ctas);
  *bytes = recon_ws_bytes(n_sub, ctas.size(), n_mu, n_red);
  return LRBMS_OK;
}

int lrbms_recon_error(lrbms_handle_t h, int32_t n_sub, const lrbms_recon_block_t* blocks_host, int64_t n_mu,
                      const double* u_h, int32_t ldu, const double* u_N, int32_t n_red, int32_t ldn, double* e, int32_t lde,
                      void* workspace, size_t workspace_bytes, void* stream) {
  LRBMS_REQUIRE(h, h && n_sub >= 0 && (n_sub == 0 || blocks_host) && n_mu >= 0 && n_red >= 0, "recon_error: bad argument");
  LRBMS_REQUIRE(h, n_mu <= INT32_MAX, "recon_error: more than 2^31 parameters");
  LRBMS_REQUIRE(h, ldu >= n_mu && lde >= n_mu && ldn >= n_red,
                "recon_error: leading dimension smaller than the batch (ldu, lde >= n_mu, ldn >= n_red)");
  int rc = check_recon_blocks(h, n_sub, blocks_host);
  if (rc) return rc;
  bool any_rows = false;
  std::vector<ReconDev> dev(n_sub);
  for (int i = 0; i < n_sub; ++i) {
    const lrbms_recon_block_t& b = blocks_host[i];
    const std::string who = "recon_error: block " + std::to_string(i) + ": ";
    LRBMS_REQUIRE(h, b.len >= 0 && b.N >= 0, who + "negative basis length");
    LRBMS_REQUIRE(h, b.N <= b.len, who + "N = " + std::to_string(b.N) + " exceeds the basis length " + std::to_string(b.len));
    LRBMS_REQUIRE(h, b.red_offset >= 0 && (int64_t)b.red_offset + b.N <= n_red, who + "coefficients outside u_N");
    LRBMS_REQUIRE(h, b.N == 0 || b.n_rows == 0 || (b.V && b.ldv >= b.len), who + "null basis or ldv < len");
    dev[i] = {b.V, b.ldv, b.row_offset, b.N, b.red_offset};
    any_rows = any_rows || b.n_rows > 0;
  }
  if (n_mu == 0 || !any_rows) return LRBMS_OK;
  LRBMS_REQUIRE(h, u_h && e && (n_red == 0 || u_N) && workspace, "recon_error: null argument");
  std::vector<CtaRange> ctas;
  recon_partition(blocks_host, n_sub, h->sm_count, &ctas);
  LRBMS_REQUIRE(h, workspace_bytes >= recon_ws_bytes(n_sub, ctas.size(), n_mu, n_red),
                "recon_error: workspace too small (see lrbms_recon_error_workspace_bytes)");
  LRBMS_CUDA_CHECK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t ldc = recon_ldc(n_mu);
  const size_t off_tab = align256(sizeof(double) * (size_t)n_red * ldc);
  const size_t off_ctas = align256(sizeof(ReconDev) * (size_t)n_sub);
  std::vector<char> table(off_ctas + sizeof(CtaRange) * ctas.size(), 0);
  std::memcpy(table.data(), dev.data(), sizeof(ReconDev) * dev.size());
  std::memcpy(table.data() + off_ctas, ctas.data(), sizeof(CtaRange) * ctas.size());
  char* w = (char*)workspace;
  LRBMS_CUDA_CHECK(h, cudaMemcpyAsync(w + off_tab, table.data(), table.size(), cudaMemcpyHostToDevice, s));
  double* ct = (double*)w;
  const ReconDev* d_blocks = (const ReconDev*)(w + off_tab);
  const CtaRange* d_ctas = (const CtaRange*)(w + off_tab + off_ctas);
  if (n_red > 0) {
    const int64_t total = (int64_t)n_red * n_mu;
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((total + 255) / 256, 8 * (int64_t)h->sm_count));
    c_t_kernel<<<grid, 256, 0, s>>>(u_N, ldn, (int)n_mu, n_red, ct, ldc);
  }
  recon_error_kernel<<<(unsigned)ctas.size(), kThreads, 0, s>>>(d_blocks, d_ctas, u_h, ldu, ct, ldc, e, lde, (int)n_mu);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  return LRBMS_OK;
}

int lrbms_segmented_form_workspace_bytes(lrbms_handle_t h, int32_t n_seg, const int32_t* seg_ptr_host, size_t* bytes) {
  LRBMS_REQUIRE(h, h && bytes && n_seg >= 0 && seg_ptr_host, "segmented_form_workspace_bytes: bad argument");
  for (int s = 0; s < n_seg; ++s)
    LRBMS_REQUIRE(h, seg_ptr_host[s] >= 0 && seg_ptr_host[s + 1] >= seg_ptr_host[s], "segmented_form_workspace_bytes: seg_ptr must be non-decreasing");
  std::vector<CtaRange> ctas;
  std::vector<int32_t> seg_cta;
  form_partition(n_seg, seg_ptr_host, h->sm_count, &ctas, &seg_cta);
  *bytes = form_ws_bytes(n_seg, ctas.size());
  return LRBMS_OK;
}

int lrbms_segmented_form(lrbms_handle_t h, int32_t n, int32_t Q, const int32_t* rowptr, const int32_t* colind,
                         const double* values, int64_t nnz, int32_t n_seg, const int32_t* seg_ptr_host, int64_t n_mu,
                         const double* theta, int32_t ldt, const double* x, int32_t ldx, double* out, int32_t ldo,
                         void* workspace, size_t workspace_bytes, void* stream) {
  LRBMS_REQUIRE(h, h && n >= 0 && nnz >= 0 && n_seg >= 0 && seg_ptr_host && n_mu >= 0, "segmented_form: bad argument");
  LRBMS_REQUIRE(h, Q >= 1, "segmented_form: Q must be at least 1");
  if (Q > kMaxQ) return lrbms_fail(h, LRBMS_ERR_UNSUPPORTED, "segmented_form: at most 4 affine operator terms are supported");
  LRBMS_REQUIRE(h, theta || Q == 1, "segmented_form: theta may only be omitted (theta = 1) for Q = 1");
  LRBMS_REQUIRE(h, !theta || ldt >= Q, "segmented_form: ldt < Q");
  LRBMS_REQUIRE(h, ldx >= n_mu && ldo >= n_mu, "segmented_form: leading dimension smaller than the batch (ldx, ldo >= n_mu)");
  for (int s = 0; s < n_seg; ++s)
    LRBMS_REQUIRE(h, seg_ptr_host[s] >= 0 && seg_ptr_host[s + 1] >= seg_ptr_host[s] && seg_ptr_host[s + 1] <= n,
                  "segmented_form: seg_ptr must be non-decreasing within [0, n]");
  if (n_mu == 0 || n_seg == 0) return LRBMS_OK;
  LRBMS_REQUIRE(h, rowptr && colind && values && x && out && workspace, "segmented_form: null argument");
  std::vector<CtaRange> ctas;
  std::vector<int32_t> seg_cta;
  form_partition(n_seg, seg_ptr_host, h->sm_count, &ctas, &seg_cta);
  LRBMS_REQUIRE(h, workspace_bytes >= form_ws_bytes(n_seg, ctas.size()),
                "segmented_form: workspace too small (see lrbms_segmented_form_workspace_bytes)");
  LRBMS_CUDA_CHECK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t off_ctas = align256(sizeof(double) * kChunk * ctas.size());
  const size_t off_seg = off_ctas + align256(sizeof(CtaRange) * ctas.size());
  std::vector<char> table(off_seg - off_ctas + sizeof(int32_t) * seg_cta.size(), 0);
  std::memcpy(table.data(), ctas.data(), sizeof(CtaRange) * ctas.size());
  std::memcpy(table.data() + (off_seg - off_ctas), seg_cta.data(), sizeof(int32_t) * seg_cta.size());
  LRBMS_CUDA_CHECK(h, cudaMemcpyAsync((char*)workspace + off_ctas, table.data(), table.size(), cudaMemcpyHostToDevice, s));
  double* part = (double*)workspace;
  const CtaRange* d_ctas = (const CtaRange*)((char*)workspace + off_ctas);
  const int32_t* d_seg = (const int32_t*)((char*)workspace + off_seg);
  const void* K = form_kernel_for_q(Q);
  int64_t ldt64 = ldt, ldx64 = ldx;
  for (int64_t m0 = 0; m0 < n_mu; m0 += kChunk) {
    int n_c = (int)std::min<int64_t>(kChunk, n_mu - m0);
    const double* th = theta ? theta + m0 * ldt : nullptr;
    const double* xm = x + m0;
    if (!ctas.empty()) {
      void* args[] = {(void*)&rowptr, (void*)&colind, (void*)&values, (void*)&nnz, (void*)&th, (void*)&ldt64,
                      (void*)&xm, (void*)&ldx64, (void*)&n_c, (void*)&d_ctas, (void*)&part};
      LRBMS_CUDA_CHECK(h, cudaLaunchKernel(K, dim3((unsigned)ctas.size()), dim3(kThreads), args, 0, s));
    }
    const int64_t total = (int64_t)n_seg * n_c;
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((total + 255) / 256, 4 * (int64_t)h->sm_count));
    segment_sum_kernel<<<grid, 256, 0, s>>>(part, d_seg, n_seg, n_c, out + m0, ldo);
    LRBMS_CUDA_CHECK(h, cudaGetLastError());
  }
  return LRBMS_OK;
}

}  // extern "C"
