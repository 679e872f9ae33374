// Context management and the GPU VectorArray backing kernels of liblrbms_sm100.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

thread_local std::string g_create_error;

int ctx_streams(lrbms_context* ctx) {
  if (!ctx->streams_ready) {
    ctx->streams_ready = true;
    bool ok = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < kSideStreams && ok; ++i)
      ok = cudaStreamCreateWithFlags(&ctx->side[i], cudaStreamNonBlocking) == cudaSuccess &&
           cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) { ctx->streams_failed = true; cudaGetLastError(); }
  }
  return (ctx->single_stream || ctx->streams_failed) ? 1 : 1 + kSideStreams;
}

void ctx_fork(lrbms_context* ctx, cudaStream_t s) {
  if (ctx_streams(ctx) == 1) return;
  cudaEventRecord(ctx->ev_fork, s);
  for (int i = 0; i < kSideStreams; ++i) cudaStreamWaitEvent(ctx->side[i], ctx->ev_fork, 0);
}

void ctx_join(lrbms_context* ctx, cudaStream_t s) {
  if (ctx_streams(ctx) == 1) return;
  for (int i = 0; i < kSideStreams; ++i) {
    cudaEventRecord(ctx->ev_join[i], ctx->side[i]);
    cudaStreamWaitEvent(s, ctx->ev_join[i], 0);
  }
}

namespace {
// test hook: every resident CTA fills its whole dynamic shared memory with quiet NaNs and holds it until all have
__global__ void poison_shared_kernel(int n_doubles) {
  extern __shared__ double poison[];
  for (int i = threadIdx.x; i < n_doubles; i += blockDim.x) poison[i] = __longlong_as_double(0x7ff8000000000000ll);
  __syncthreads();
  if (poison[n_doubles - 1] == 0.0) printf("unreachable\n");    // keeps the stores alive
}
}  // namespace

extern "C" {

int lrbms_version(void) { return LRBMS_VERSION; }

int lrbms_debug_poison_shared(lrbms_handle_t h, void* stream) {
  LRBMS_REQUIRE(h, h != nullptr, "lrbms_debug_poison_shared: null handle");
  LRBMS_CUDA_CHECK(h, cudaSetDevice(h->device));
  const int bytes = h->max_smem_optin - 1024;
  LRBMS_CUDA_CHECK(h, cudaFuncSetAttribute(poison_shared_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  poison_shared_kernel<<<4 * h->sm_count, 256, bytes, (cudaStream_t)stream>>>(bytes / 8);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  return LRBMS_OK;
}

int lrbms_set_option(lrbms_handle_t h, int32_t option, int32_t value) {
  LRBMS_REQUIRE(h, h != nullptr, "lrbms_set_option: null handle");
  switch (option) {
    case LRBMS_OPT_SINGLE_STREAM: h->single_stream = value != 0; return LRBMS_OK;
    case LRBMS_OPT_PCG_MULTI_LAUNCH: h->single_launch_pcg_off = value != 0; return LRBMS_OK;
    default: return lrbms_fail(h, LRBMS_ERR_INVALID, "lrbms_set_option: unknown option");
  }
}

int lrbms_create(int device, lrbms_handle_t* out) {
  if (!out) return lrbms_fail(nullptr, LRBMS_ERR_INVALID, "lrbms_create: out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return lrbms_fail(nullptr, LRBMS_ERR_NO_DEVICE,
                      std::string("no CUDA device available (") + cudaGetErrorString(e) +
                          "); liblrbms_sm100 has no CPU fallback");
  if (device < 0 || device >= count) return lrbms_fail(nullptr, LRBMS_ERR_INVALID, "lrbms_create: bad device index");
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return lrbms_fail(nullptr, LRBMS_ERR_CUDA, cudaGetErrorString(e));
  if (prop.major != 10)
    return lrbms_fail(nullptr, LRBMS_ERR_NO_DEVICE,
                      "device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                          "; this library is built for sm_100a only");
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return lrbms_fail(nullptr, LRBMS_ERR_CUDA, cudaGetErrorString(e));
  {
    // keep freed plan memory in the default pool (see plan_alloc)
    cudaMemPool_t pool = nullptr;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess && pool) {
      unsigned long long keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
  }
  lrbms_context* ctx = new lrbms_context();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
  *out = ctx;
  return LRBMS_OK;
}

int lrbms_destroy(lrbms_handle_t h) {
  if (h && h->streams_ready) {
    for (int i = 0; i < kSideStreams; ++i) {
      if (h->side[i]) cudaStreamDestroy(h->side[i]);
      if (h->ev_join[i]) cudaEventDestroy(h->ev_join[i]);
    }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  }
  delete h;
  return LRBMS_OK;
}

const char* lrbms_last_error(lrbms_handle_t h) { return h ? h->last_error.c_str() : g_create_error.c_str(); }

int lrbms_device_sm_count(lrbms_handle_t h, int* out) {
  if (!h || !out) return LRBMS_ERR_INVALID;
  *out = h->sm_count;
  return LRBMS_OK;
}

int lrbms_plan_run(lrbms_plan_t plan, void* stream) {
  if (!plan) return LRBMS_ERR_INVALID;
  return plan->run(stream);
}

int lrbms_plan_destroy(lrbms_plan_t plan) {
  if (!plan) return LRBMS_OK;
  // the plan's buffers go back to the pool in stream order; work that still uses them may sit on any stream
  if (plan->ctx) cudaSetDevice(plan->ctx->device);
  if (!plan->device_allocs.empty()) cudaDeviceSynchronize();
  for (void* p : plan->device_allocs) cudaFreeAsync(p, (cudaStream_t)0);
  delete plan;
  return LRBMS_OK;
}

int lrbms_plan_info(lrbms_plan_t plan, int32_t what, double* out) {
  if (!plan || !out) return LRBMS_ERR_INVALID;
  if (what == 2 || what == 3 || what == 5) plan->ensure_info();
  switch (what) {
    case 0: *out = plan->info_launches; break;
    case 1: *out = plan->info_ctas; break;
    case 2: *out = plan->info_bytes; break;
    case 3: *out = plan->info_flops; break;
    case 4: *out = (double)plan->device_bytes; break;
    case 5: *out = plan->info_bytes_survey; break;
    case 6: *out = plan->info_solver; break;
    case 7: *out = plan->info_solve_flops; break;
    case 8: *out = plan->info_half_bandwidth; break;
    case 9: *out = plan->info_est_tmu; break;
    default: return lrbms_fail(plan->ctx, LRBMS_ERR_INVALID, "lrbms_plan_info: unknown selector");
  }
  return LRBMS_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------------
//  Incremental re-projection: assembly of the new reduced blocks from the previous ones and the narrow projections of
//  the appended basis vectors (one CTA per block).
// ------------------------------------------------------------------------------------------------------
namespace {
__global__ void remap_blocks_kernel(const lrbms_remap_desc_t* __restrict__ descs) {
  const lrbms_remap_desc_t D = descs[blockIdx.x];
  const int total = D.NL * D.NR;
  for (int e = threadIdx.x; e < total; e += blockDim.x) {
    const int r = e / D.NR, c = e - r * D.NR;
    const int rm = D.row_map[r], cm = D.col_map[c];
    double v;
    if (cm < 0) v = D.cols_new[(int64_t)r * D.n_cn + (-cm - 1)];
    else if (rm < 0) v = D.rows_new ? D.rows_new[(int64_t)c * D.n_rn + (-rm - 1)] : D.cols_new[(int64_t)c * D.n_cn + (-rm - 1)];
    else v = D.prev[(int64_t)rm * D.pNR + cm];
    D.dst[e] = v;
  }
}
}  // namespace

extern "C" int lrbms_remap_blocks(lrbms_handle_t h, int32_t n, const lrbms_remap_desc_t* descs_host, void* stream) {
  LRBMS_REQUIRE(h, h && (n == 0 || descs_host) && n >= 0, "remap_blocks: bad argument");
  if (n == 0) return LRBMS_OK;
  LRBMS_CUDA_CHECK(h, cudaSetDevice(h->device));
  for (int i = 0; i < n; ++i) {
    const auto& d = descs_host[i];
    LRBMS_REQUIRE(h, d.dst && d.row_map && d.col_map && d.NL >= 0 && d.NR >= 0, "remap_blocks: null pointer in descriptor");
  }
  cudaStream_t s = (cudaStream_t)stream;
  lrbms_remap_desc_t* dd = nullptr;
  LRBMS_CUDA_CHECK(h, cudaMallocAsync((void**)&dd, sizeof(lrbms_remap_desc_t) * n, s));
  LRBMS_CUDA_CHECK(h, cudaMemcpyAsync(dd, descs_host, sizeof(lrbms_remap_desc_t) * n, cudaMemcpyHostToDevice, s));
  LRBMS_CUDA_CHECK(h, cudaStreamSynchronize(s));        // descs_host may be released by the caller after return
  remap_blocks_kernel<<<n, 256, 0, s>>>(dd);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  LRBMS_CUDA_CHECK(h, cudaFreeAsync(dd, s));
  return LRBMS_OK;
}

// ------------------------------------------------------------------------------------------------------
//  Peer-memory exchange of the sharded offline results: every rank stores its contiguous region of reduced blocks
//  straight into the other GPUs' staging buffers over NVLink (mapped peer pointers), or -- when the NVSwitch multicast
//  object exists -- once into the multicast address, which the switch replicates to every GPU.  The caller orders the
//  stores against the readers with a device-side barrier of the symmetric-memory signal pads afterwards.
// ------------------------------------------------------------------------------------------------------
namespace {
struct PeerTargets {
  unsigned long long dst[LRBMS_MAX_PEERS];
  int n, multicast;
};

__global__ void __launch_bounds__(256) peer_push_kernel(const int4* __restrict__ src, int64_t n16, PeerTargets T) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) {
    const int4 v = src[i];
    if (T.multicast) {
      asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(T.dst[0] + 16ull * (unsigned long long)i),
                   "f"(__int_as_float(v.x)), "f"(__int_as_float(v.y)), "f"(__int_as_float(v.z)), "f"(__int_as_float(v.w))
                   : "memory");
    } else {
#pragma unroll 1
      for (int d = 0; d < T.n; ++d) *reinterpret_cast<int4*>(T.dst[d] + 16ull * (unsigned long long)i) = v;
    }
  }
}
}  // namespace

extern "C" int lrbms_peer_push(lrbms_handle_t h, const void* src, int64_t n_bytes, int32_t n_dst, const uint64_t* dst_host,
                               int32_t multicast, void* stream) {
  LRBMS_REQUIRE(h, h && n_bytes >= 0 && n_dst >= 0 && n_dst <= LRBMS_MAX_PEERS && (n_dst == 0 || dst_host),
                "peer_push: bad argument");
  if (n_bytes == 0 || n_dst == 0) return LRBMS_OK;
  LRBMS_REQUIRE(h, src && n_bytes % 16 == 0 && ((uintptr_t)src & 15) == 0, "peer_push: the region must be 16-byte aligned and sized");
  LRBMS_REQUIRE(h, !multicast || n_dst == 1, "peer_push: a multicast push has exactly one (multicast) destination");
  PeerTargets T{};
  T.n = n_dst;
  T.multicast = multicast ? 1 : 0;
  for (int d = 0; d < n_dst; ++d) {
    LRBMS_REQUIRE(h, dst_host[d] && (dst_host[d] & 15) == 0, "peer_push: unaligned or null destination");
    T.dst[d] = dst_host[d];
  }
  LRBMS_CUDA_CHECK(h, cudaSetDevice(h->device));
  const int64_t n16 = n_bytes / 16;
  const int grid = (int)std::min<int64_t>((n16 + 255) / 256, (int64_t)h->sm_count * 8);
  peer_push_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const int4*>(src), n16, T);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  return LRBMS_OK;
}

// ------------------------------------------------------------------------------------------------------
//  VectorArray kernels.  Arrays are dof-major (dim x ld); a "row" is one dof across all vectors, so every
//  kernel walks rows with consecutive threads on consecutive vectors -> coalesced for ld == len.
// ------------------------------------------------------------------------------------------------------
namespace {

constexpr int kMaxAlpha = 256;
struct AlphaPack { double a[kMaxAlpha]; };

__global__ void va_scal_kernel(int64_t dim, int len, AlphaPack alpha, int n_alpha, double* __restrict__ y, int ldy) {
  int64_t total = dim * (int64_t)len;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t d = idx / len;
    int a = (int)(idx - d * len);
    y[d * ldy + a] *= alpha.a[n_alpha == 1 ? 0 : a];
  }
}

__global__ void va_axpy_kernel(int64_t dim, int len, AlphaPack alpha, int n_alpha, const double* __restrict__ x, int ldx,
                               int len_x, double* __restrict__ y, int ldy) {
  int64_t total = dim * (int64_t)len;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t d = idx / len;
    int a = (int)(idx - d * len);
    y[d * ldy + a] += alpha.a[n_alpha == 1 ? 0 : a] * x[d * ldx + (len_x == 1 ? 0 : a)];
  }
}

// one CTA per chunk of dofs; partial sums reduced through shared memory then atomically (deterministic enough for
// norms: the order over chunks is fixed by using a two-pass scheme instead of atomics)
__global__ void va_pairwise_dot_partial(int64_t dim, int len, const double* __restrict__ x, int ldx,
                                        const double* __restrict__ y, int ldy, double* __restrict__ partial) {
  // thread (a = threadIdx.x % len_pad, lane row = threadIdx.x / len_pad)
  extern __shared__ double sm[];
  int rows_per_pass = blockDim.x / len;
  int a = threadIdx.x % len;
  int r = threadIdx.x / len;
  double acc = 0.0;
  if (r < rows_per_pass) {
    for (int64_t d = (int64_t)blockIdx.x * rows_per_pass + r; d < dim; d += (int64_t)gridDim.x * rows_per_pass)
      acc += x[d * ldx + a] * y[d * ldy + a];
  }
  sm[threadIdx.x] = (r < rows_per_pass) ? acc : 0.0;
  __syncthreads();
  if (threadIdx.x < len) {
    double s = 0.0;
    for (int rr = 0; rr < rows_per_pass; ++rr) s += sm[rr * len + threadIdx.x];
    partial[(int64_t)blockIdx.x * len + threadIdx.x] = s;
  }
}

__global__ void va_reduce_partials(int n_part, int len, const double* __restrict__ partial, double* __restrict__ out) {
  int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= len) return;
  double s = 0.0;
  for (int p = 0; p < n_part; ++p) s += partial[(int64_t)p * len + a];
  out[a] = s;
}

// y[d, j] = sum_a x[d, a] * C[a, j]; one warp per dof row, coefficient matrix staged in shared memory
__global__ void va_lincomb_kernel(int64_t dim, int len, int n_out, const double* __restrict__ x, int ldx,
                                  const double* __restrict__ coeff, int ldc, double* __restrict__ y, int ldy) {
  extern __shared__ double sC[];   // len x n_out
  for (int i = threadIdx.x; i < len * n_out; i += blockDim.x) sC[i] = coeff[(i / n_out) * (int64_t)ldc + (i % n_out)];
  __syncthreads();
  int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int64_t d = (int64_t)blockIdx.x * nw + warp; d < dim; d += (int64_t)gridDim.x * nw) {
    const double* xr = x + d * ldx;
    for (int j = lane; j < n_out; j += 32) {
      double acc = 0.0;
      for (int a = 0; a < len; ++a) acc += xr[a] * sC[a * n_out + j];
      y[d * ldy + j] = acc;
    }
  }
}

struct ColPack { int c[kMaxAlpha]; };
__global__ void va_copy_cols_kernel(int64_t dim, int n_cols, ColPack src, int identity, const double* __restrict__ x,
                                    int ldx, double* __restrict__ y, int ldy, int dst0) {
  int64_t total = dim * (int64_t)n_cols;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t d = idx / n_cols;
    int k = (int)(idx - d * n_cols);
    y[d * ldy + dst0 + k] = x[d * ldx + (identity ? k : src.c[k])];
  }
}

// tiled transpose: in (len x dim, row-major) -> out (dim x ld)
__global__ void va_transpose_kernel(int64_t rows_in, int64_t cols_in, const double* __restrict__ in, int64_t ld_in,
                                    double* __restrict__ out, int64_t ld_out) {
  __shared__ double tile[32][33];
  int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int64_t r = r0 + j, c = c0 + threadIdx.x;
    if (r < rows_in && c < cols_in) tile[j][threadIdx.x] = in[r * ld_in + c];
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int64_t c = c0 + j, r = r0 + threadIdx.x;   // out[c][r]
    if (r < rows_in && c < cols_in) out[c * ld_out + r] = tile[threadIdx.x][j];
  }
}

inline int grid_for(int64_t total, int block, int sm_count) {
  int64_t g = (total + block - 1) / block;
  int64_t cap = (int64_t)sm_count * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

extern "C" {

int lrbms_va_scal(lrbms_handle_t h, int64_t dim, int32_t len, const double* alpha_host, int32_t n_alpha, double* y,
                  int32_t ldy, void* stream) {
  LRBMS_REQUIRE(h, h && y && alpha_host, "va_scal: null argument");
  LRBMS_REQUIRE(h, (n_alpha == 1 || n_alpha == len) && len <= kMaxAlpha, "va_scal: n_alpha must be 1 or len (<= 256)");
  if (dim == 0 || len == 0) return LRBMS_OK;
  AlphaPack ap;
  for (int i = 0; i < n_alpha; ++i) ap.a[i] = alpha_host[i];
  va_scal_kernel<<<grid_for(dim * len, 256, h->sm_count), 256, 0, (cudaStream_t)stream>>>(dim, len, ap, n_alpha, y, ldy);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  return LRBMS_OK;
}

int lrbms_va_axpy(lrbms_handle_t h, int64_t dim, int32_t len, const double* alpha_host, int32_t n_alpha, const double* x,
                  int32_t ldx, int32_t len_x, double* y, int32_t ldy, void* stream) {
  LRBMS_REQUIRE(h, h && x && y && alpha_host, "va_axpy: null argument");
  LRBMS_REQUIRE(h, (n_alpha == 1 || n_alpha == len) && len <= kMaxAlpha, "va_axpy: n_alpha must be 1 or len (<= 256)");
  LRBMS_REQUIRE(h, len_x == 1 || len_x == len, "va_axpy: len(x) must be 1 or len(y)");
  if (dim == 0 || len == 0) return LRBMS_OK;
  AlphaPack ap;
  for (int i = 0; i < n_alpha; ++i) ap.a[i] = alpha_host[i];
  va_axpy_kernel<<<grid_for(dim * len, 256, h->sm_count), 256, 0, (cudaStream_t)stream>>>(dim, len, ap, n_alpha, x, ldx,
                                                                                          len_x, y, ldy);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  return LRBMS_OK;
}

int lrbms_va_pairwise_dot(lrbms_handle_t h, int64_t dim, int32_t len, const double* x, int32_t ldx, const double* y,
                          int32_t ldy, double* out, void* stream) {
  LRBMS_REQUIRE(h, h && x && y && out, "va_pairwise_dot: null argument");
  LRBMS_REQUIRE(h, len >= 1 && len <= 256, "va_pairwise_dot: len must be in [1, 256]");
  const int block = 256;
  int rows_per_pass = block / len;
  int n_part = (int)((dim + rows_per_pass - 1) / rows_per_pass);
  if (n_part > h->sm_count * 4) n_part = h->sm_count * 4;
  if (n_part < 1) n_part = 1;
  double* partial = nullptr;
  LRBMS_CUDA_CHECK(h, cudaMallocAsync((void**)&partial, (size_t)n_part * len * sizeof(double), (cudaStream_t)stream));
  va_pairwise_dot_partial<<<n_part, block, block * sizeof(double), (cudaStream_t)stream>>>(dim, len, x, ldx, y, ldy, partial);
  va_reduce_partials<<<(len + 127) / 128, 128, 0, (cudaStream_t)stream>>>(n_part, len, partial, out);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  LRBMS_CUDA_CHECK(h, cudaFreeAsync(partial, (cudaStream_t)stream));
  return LRBMS_OK;
}

int lrbms_va_lincomb(lrbms_handle_t h, int64_t dim, int32_t len, int32_t n_out, const double* x, int32_t ldx,
                     const double* coeff, int32_t ldc, double* y, int32_t ldy, void* stream) {
  LRBMS_REQUIRE(h, h && x && y && coeff, "va_lincomb: null argument");
  size_t smem = (size_t)len * n_out * sizeof(double);
  LRBMS_REQUIRE(h, smem <= 48 * 1024, "va_lincomb: len * n_out too large for one call (chunk n_out on the host side)");
  if (dim == 0 || n_out == 0) return LRBMS_OK;
  int grid = (int)((dim + 7) / 8);
  if (grid > h->sm_count * 8) grid = h->sm_count * 8;
  va_lincomb_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(dim, len, n_out, x, ldx, coeff, ldc, y, ldy);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  return LRBMS_OK;
}

int lrbms_va_copy_cols(lrbms_handle_t h, int64_t dim, int32_t n_cols, const int32_t* src_host, const double* x, int32_t ldx,
                       double* y, int32_t ldy, int32_t dst0, void* stream) {
  LRBMS_REQUIRE(h, h && x && y, "va_copy_cols: null argument");
  LRBMS_REQUIRE(h, n_cols <= kMaxAlpha, "va_copy_cols: at most 256 columns per call");
  if (dim == 0 || n_cols == 0) return LRBMS_OK;
  ColPack cp;
  if (src_host) for (int i = 0; i < n_cols; ++i) cp.c[i] = src_host[i];
  va_copy_cols_kernel<<<grid_for(dim * n_cols, 256, h->sm_count), 256, 0, (cudaStream_t)stream>>>(
      dim, n_cols, cp, src_host ? 0 : 1, x, ldx, y, ldy, dst0);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  return LRBMS_OK;
}

int lrbms_va_transpose_in(lrbms_handle_t h, int64_t dim, int32_t len, const double* rowmajor_len_dim, double* dofmajor,
                          int32_t ld, void* stream) {
  LRBMS_REQUIRE(h, h && rowmajor_len_dim && dofmajor, "va_transpose_in: null argument");
  if (dim == 0 || len == 0) return LRBMS_OK;
  dim3 grid((unsigned)((dim + 31) / 32), (unsigned)((len + 31) / 32)), block(32, 8);
  va_transpose_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(len, dim, rowmajor_len_dim, dim, dofmajor, ld);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  return LRBMS_OK;
}

int lrbms_va_transpose_out(lrbms_handle_t h, int64_t dim, int32_t len, const double* dofmajor, int32_t ld,
                           double* rowmajor_len_dim, void* stream) {
  LRBMS_REQUIRE(h, h && rowmajor_len_dim && dofmajor, "va_transpose_out: null argument");
  if (dim == 0 || len == 0) return LRBMS_OK;
  dim3 grid((unsigned)((len + 31) / 32), (unsigned)((dim + 31) / 32)), block(32, 8);
  va_transpose_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(dim, len, dofmajor, ld, rowmajor_len_dim, dim);
  LRBMS_CUDA_CHECK(h, cudaGetLastError());
  return LRBMS_OK;
}

}  // extern "C"
