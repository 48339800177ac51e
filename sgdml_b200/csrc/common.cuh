// Shared helpers for the sgdml_b200 CUDA sources (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/sgdml_b200.h"

namespace sgdml {

// ------------------------------------------------------------------ error plumbing
void set_last_error(const std::string& msg);
int fail_cuda(cudaError_t e, const char* what, const char* file, int line);
int fail_arg(const char* what);

#define SG_CUDA(expr)                                                        \
  do {                                                                       \
    cudaError_t _e = (expr);                                                 \
    if (_e != cudaSuccess) return ::sgdml::fail_cuda(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define SG_TRY(expr)            \
  do {                          \
    int _rc = (expr);           \
    if (_rc != 0) return _rc;   \
  } while (0)

#define SG_ARG(cond)                                    \
  do {                                                  \
    if (!(cond)) return ::sgdml::fail_arg(#cond);       \
  } while (0)

// Checks that a CUDA device is present (the product has no CPU fallback).
int require_device();

// ------------------------------------------------------------------ host/device staging
bool is_device_ptr(const void* p);

// RAII staging buffer: presents a device view of a user pointer that may live on the host.
// in:  copy host->device on construction when the user pointer is a host pointer
// out: copy device->host in finish() when the user pointer is a host pointer
// The device buffers come from a small per-thread pool: cudaMalloc + cudaFree cost ~10 ms each in a
// process that holds tens of GB (measured: 4 pairs per preconditioner application = 86 ms), which
// dominated calls made once per CG iteration.  On destruction the stream the buffer was used on is
// synchronised (what the implicit synchronisation of cudaFree used to guarantee) and the buffer is
// kept for the next call.
class Staged {
 public:
  Staged() {}
  ~Staged();
  Staged(const Staged&) = delete;
  Staged& operator=(const Staged&) = delete;
  // Returns 0 on success.  user may be NULL (then dev() is NULL).
  int init(const void* user, size_t bytes, bool copy_in, cudaStream_t s);
  void* dev() const { return dev_; }
  bool staged() const { return owns_; }
  // For outputs: copies back to the host pointer (async on s).
  int finish(cudaStream_t s);

 private:
  void* dev_ = nullptr;
  void* user_ = nullptr;
  size_t bytes_ = 0;
  size_t cap_ = 0;
  int dev_id_ = 0;
  cudaStream_t stream_ = nullptr;
  bool owns_ = false;
};

// Persistent device workspaces for calls that run once per training run or more often (the Cholesky panel
// workspace is 516 MB at BASELINE config 2; a cudaMalloc / cudaFree pair of that size costs milliseconds and
// synchronises the device).  One buffer per (device, slot), grown on demand, kept until
// sgdml_b200_release_workspaces().  The caller must have finished with the buffer (stream synchronised) before the
// next ws_get of the same slot -- true for every user: they all synchronise before returning.
enum WsSlot { WS_POTRF_W0 = 0, WS_POTRF_W1 = 1, WS_OZ_PLANES = 2, WS_OZ_EXPS = 3, WS_POTRF_INFO = 4, WS_SOLVE_TMP = 5,
              WS_ASM_DPERM = 6, WS_ASM_APERM = 7, WS_ASM_APINV = 8, WS_ASM_JPTS = 9, WS_ASM_DEST = 10, WS_ASM_SLABS = 11,
              WS_SLOT_COUNT = 12 };
int ws_get(int slot, size_t bytes, void** out);

// Device-block cache for the predictor's model arrays and per-batch workspaces: `GDMLTrain.train` creates and destroys a
// predictor of the same shape every run (integration constant), and on some hosts a cudaMalloc / cudaFree pair next to
// a 32 GB K buffer costs 5-15 ms (measured: 0.2-0.5 s of a 1.3 s training run on such a box, 3 ms on others).
// cached_free keeps a block (exact-size reuse, at most 8 GB in total); the CALLER makes sure no kernel still uses it
// (cudaFree's implicit synchronisation is gone).  sgdml_b200_release_workspaces() empties the cache.
cudaError_t cached_malloc_bytes(void** p, size_t bytes);
cudaError_t cached_free(void* p);
void cache_release_all();
template <class T>
inline cudaError_t cached_malloc(T** p, size_t bytes) {
  return cached_malloc_bytes(reinterpret_cast<void**>(p), bytes);
}

inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

int num_sms();

// ------------------------------------------------------------------ launch accounting / profiling
// Kernel families (ids of sgdml_b200_profile_get).
enum KernelId { KID_PREDICT_MAIN = 0, KID_PREDICT_AUX = 1, KID_ASSEMBLE = 2, KID_GEMM = 3, KID_POTF2 = 4,
                KID_TRSM = 5, KID_TRSV = 6, KID_DESC = 7, KID_MISC = 8, KID_HESSIAN = 9,
                KID_COUNT = 10 };
void count_launch(int kid, int n = 1);
// When profiling is enabled, ProfScope records CUDA events around a launch sequence on `s`
// and adds the elapsed device time to the family's total (synchronises at scope exit).
bool profiling_enabled();
class ProfScope {
 public:
  ProfScope(int kid, cudaStream_t s);
  ~ProfScope();

 private:
  int kid_;
  cudaStream_t s_;
  cudaEvent_t e0_ = nullptr, e1_ = nullptr;
};

// ------------------------------------------------------------------ device helpers
#ifdef __CUDACC__

// FP64 tensor-pipe MMA, D(8x8) += A(8x4, row) * B(4x8, col).
// Fragment layouts (PTX ISA, mma.m8n8k4 .f64): lane l holds
//   a = A[l/4][l%4],  b = B[l%4][l/4],  c0,c1 = C[l/4][2*(l%4) + {0,1}].
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// ---- mbarrier + 1-D bulk async copy (TMA engine, SASS UBLKCP)
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// global -> shared bulk copy, completion signalled on an mbarrier (bytes multiple of 16,
// both addresses 16-byte aligned).
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---- Ampere-style cp.async (SASS LDGSTS), 16 bytes
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async16_pred(void* smem_dst, const void* gmem_src, bool pred) {
  // src-size 0 => zero fill
  int sz = pred ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(sz)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

#endif  // __CUDACC__

}  // namespace sgdml
