// Shared internals of liblrbms_sm100: context / plan structs, error plumbing, FP64 tensor-core primitive.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/lrbms_sm100.h"

constexpr int kSideStreams = 3;

struct lrbms_context {
  int device = -1;
  int sm_count = 0;
  int max_smem_optin = 0;
  std::string last_error;
  // side streams of the offline plans: the launches of one plan run (one per tile-shape bucket) are independent, so they
  // are spread over the caller's stream and these and joined again before the plan returns (lrbms_set_option(LRBMS_OPT_SINGLE_STREAM, 1): off)
  bool streams_ready = false, single_stream = false, streams_failed = false;
  bool single_launch_pcg_off = false;   // LRBMS_OPT_PCG_MULTI_LAUNCH: three launches per CG iteration instead of the cooperative kernel
  cudaStream_t side[kSideStreams] = {};
  cudaEvent_t ev_fork = nullptr, ev_join[kSideStreams] = {};
};

// lazily creates the side streams; returns the number of streams a plan run may use (1 = caller's stream only)
int ctx_streams(lrbms_context* ctx);
// side streams wait for everything enqueued on `s` so far / `s` waits for everything enqueued on the side streams
void ctx_fork(lrbms_context* ctx, cudaStream_t s);
void ctx_join(lrbms_context* ctx, cudaStream_t s);
inline cudaStream_t ctx_stream(lrbms_context* ctx, cudaStream_t s, int k, int n_streams) {
  const int i = k % n_streams;
  return i == 0 ? s : ctx->side[i - 1];
}

enum PlanKind { PLAN_SPMM = 1, PLAN_PROJECT = 2, PLAN_ONLINE = 3 };

struct lrbms_plan {
  lrbms_context* ctx = nullptr;
  PlanKind kind;
  std::vector<void*> device_allocs;   // freed in lrbms_plan_destroy
  size_t device_bytes = 0;
  double info_launches = 0, info_ctas = 0, info_bytes = 0, info_flops = 0, info_bytes_survey = 0;
  double info_solver = 0, info_solve_flops = 0, info_half_bandwidth = 0;   // online plans only
  double info_est_tmu = 0;            // online plans with an estimator: parameters per estimator CTA
  virtual ~lrbms_plan() {}
  virtual int run(void* stream) = 0;
  virtual void ensure_info() {}       // byte / flop accounting is computed on first request, not at plan creation
};

// Opens a kernel's dynamic shared-memory limit to all the device allows one block beside the kernel's own static shared
// memory, and returns that static size. The limit is an attribute of the function on the current device, shared by every
// plan: set to one plan's byte count, it would make the next launch of a larger plan that is still alive fail. It does not
// change occupancy, which follows the bytes a launch asks for.
inline cudaError_t lrbms_open_dynamic_smem(const lrbms_context* ctx, const void* fn, size_t* static_bytes = nullptr) {
  cudaFuncAttributes fa;
  cudaError_t e = cudaFuncGetAttributes(&fa, fn);
  if (e != cudaSuccess) return e;
  if (static_bytes) *static_bytes = fa.sharedSizeBytes;
  return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->max_smem_optin - (int)fa.sharedSizeBytes);
}

extern thread_local std::string g_create_error;

inline int lrbms_fail(lrbms_context* ctx, int code, const std::string& msg) {
  if (ctx) ctx->last_error = msg; else g_create_error = msg;
  return code;
}

#define LRBMS_CUDA_CHECK(ctx, expr)                                                                  \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess) {                                                                         \
      return lrbms_fail((ctx), LRBMS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));  \
    }                                                                                                \
  } while (0)

#define LRBMS_REQUIRE(ctx, cond, msg)                                             \
  do {                                                                            \
    if (!(cond)) return lrbms_fail((ctx), LRBMS_ERR_INVALID, std::string(msg));   \
  } while (0)

// Allocate device memory owned by a plan.
template <typename T>
inline int plan_alloc(lrbms_plan* p, T** out, size_t count) {
  void* ptr = nullptr;
  size_t bytes = (count ? count : 1) * sizeof(T);
  // stream-ordered allocation from the device's default pool (its release threshold is raised in lrbms_create): the plans
  // of successive reductions reuse the pooled blocks instead of paying a synchronising cudaMalloc / cudaFree each
  // (a C2 projection plan owns ~200 scratch arrays; plain cudaMalloc made plan creation take 0.2 ... 2 s)
  cudaError_t e = cudaMallocAsync(&ptr, bytes, (cudaStream_t)0);
  if (e != cudaSuccess) return lrbms_fail(p->ctx, LRBMS_ERR_ALLOC, std::string("cudaMallocAsync: ") + cudaGetErrorString(e));
  p->device_allocs.push_back(ptr);
  p->device_bytes += bytes;
  *out = reinterpret_cast<T*>(ptr);
  return 0;
}

template <typename T>
inline int plan_upload(lrbms_plan* p, T** out, const std::vector<T>& host) {
  int rc = plan_alloc(p, out, host.size());
  if (rc) return rc;
  if (!host.empty()) {
    cudaError_t e = cudaMemcpy(*out, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return lrbms_fail(p->ctx, LRBMS_ERR_CUDA, std::string("cudaMemcpy H2D: ") + cudaGetErrorString(e));
  }
  return 0;
}

#ifdef __CUDACC__
// D(8x8) += A(8x4, row) * B(4x8, col), FP64 tensor core (SASS: DMMA.8x8x4).
// lane = 4*g + t:  a = A[g][t],  b = B[t][g],  d0 = D[g][2t], d1 = D[g][2t+1].
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem_src));
}
// copies with zero fill: src_bytes (<= size) bytes are read, the rest of the destination is zeroed; src must be a valid
// address even when src_bytes == 0
__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* gmem_src, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem_src), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async8_zfill(void* smem_dst, const void* gmem_src, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(gmem_src), "r"(src_bytes));
}
// ---- bulk asynchronous copy (TMA engine, SASS UBLKCP) with mbarrier completion
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes)
               : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completes on `bar`
__device__ __forceinline__ void bulk_copy_g2s(void* smem_dst, const void* gmem_src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   (unsigned)__cvta_generic_to_shared(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  unsigned ok;
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok)
                 : "r"(a), "r"(parity)
                 : "memory");
  } while (!ok);
}
// generic-proxy accesses to shared memory before this point are ordered before later async-proxy (bulk copy) accesses
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
// the same for every state space: earlier generic-proxy stores to *global* memory (e.g. a factor written with st.global)
// are ordered before later bulk copies that read them back through the async proxy
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }
#endif
