// common.cuh -- shared helpers for the sm_100a kernels behind include/mrx.h.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/mrx.h"

namespace mrx {

// ---------------------------------------------------------------- host-side errors
void set_error(const char *fmt, ...);

#define MRX_CHECK_ARG(cond, ...)                 \
  do {                                           \
    if (!(cond)) {                               \
      ::mrx::set_error(__VA_ARGS__);             \
      return MRX_E_INVALID;                      \
    }                                            \
  } while (0)

#define MRX_CHECK_SUPPORTED(cond, ...)           \
  do {                                           \
    if (!(cond)) {                               \
      ::mrx::set_error(__VA_ARGS__);             \
      return MRX_E_UNSUPPORTED;                  \
    }                                            \
  } while (0)

#define MRX_CUDA(call)                                                         \
  do {                                                                         \
    cudaError_t e_ = (call);                                                   \
    if (e_ != cudaSuccess) {                                                   \
      ::mrx::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                       __FILE__, __LINE__);                                    \
      return MRX_E_CUDA;                                                       \
    }                                                                          \
  } while (0)

#define MRX_LAUNCH_CHECK(name)                                                 \
  do {                                                                         \
    cudaError_t e_ = cudaGetLastError();                                       \
    if (e_ != cudaSuccess) {                                                   \
      ::mrx::set_error("launch of %s failed: %s", name, cudaGetErrorString(e_)); \
      return MRX_E_CUDA;                                                       \
    }                                                                          \
  } while (0)

// ---------------------------------------------------------------- host-side launch constants
constexpr int kMaxDevices = 64;

struct DevInfo {
  int device, sms, max_smem_optin;
};
// SM count / opt-in shared memory of the current device, queried once per device.
int current_device_info(DevInfo *out);

// Remembers, per device, the dynamic shared-memory size a kernel has been opted into, so that
// cudaFuncSetAttribute runs when the requirement grows, not on every launch.
struct SmemCache {
  int set[kMaxDevices];
};
int ensure_dynamic_smem(const void *func, SmemCache *cache, int device, int bytes);

// Exclusive scan of d[0..n) in place on `stream`, d[n] = the total (one CTA; rle.cu).
int exclusive_scan_i64(long long *d, int n, cudaStream_t stream);

// ---------------------------------------------------------------- device: PTX wrappers
#if defined(__CUDACC__)

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count)
               : "memory");
}

__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// arrive (count 1) and add `bytes` to the transaction count the phase waits for
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}

// add `bytes` to the transaction count of the current phase without arriving
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}

// plain arrive (count 1), release semantics at CTA scope
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// named barrier among `nthreads` threads (id 1..15; 0 is __syncthreads)
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}

// ---- variants taking 32-bit shared-window addresses (no generic->shared conversion per call)
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_expect_tx_a(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}

// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase
// completes (or the hint elapses) instead of spinning through the issue slots
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
  uint32_t done;
#pragma unroll 1
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(bar), "r"(parity), "r"(20000u)
        : "memory");
  } while (!done);
}

// one try_wait with an explicit suspend-time hint (ns); returns whether the phase completed
__device__ __forceinline__ bool mbar_try_wait_a(uint32_t bar, uint32_t parity, uint32_t hint_ns) {
  uint32_t done;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(done)
      : "r"(bar), "r"(parity), "r"(hint_ns)
      : "memory");
  return done != 0;
}

__device__ __forceinline__ void bulk_g2s_a(uint32_t smem_dst, const void *gmem_src, uint32_t bytes,
                                           uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_dst),
      "l"(gmem_src), "r"(bytes), "r"(bar)
      : "memory");
}

// 1-D TMA: global -> shared, completion reported to an mbarrier (SASS: UBLKCP).
// dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes,
                                         uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// 1-D TMA: shared -> global, tracked by the bulk async-group of the issuing thread.
__device__ __forceinline__ void bulk_s2g(void *gmem_dst, const void *smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void bulk_commit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}

// wait until the sources of all but the newest N committed bulk groups have been read
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

template <int N>
__device__ __forceinline__ void bulk_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// make generic-proxy writes to shared memory visible to the async proxy (TMA)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// Exact source coordinate of the half-pixel-centre resize (a4):
//   src = (dst + 0.5) * in/out - 0.5 = (in*(2*dst+1) - out) / (2*out)
// returned as i0 = floor(src) in [-1, in-1] and the fractional part in [0,1) rounded
// once to fp32.  All integer quantities are < 2^24 so the float conversions are exact.
struct SrcCoord {
  int i0;
  float w;
};

__device__ __forceinline__ SrcCoord src_coord(int dst, int in, int out, float inv_2out) {
  const int D = 2 * out;
  const int A = in * (2 * dst + 1) - out;
  int i0 = __float2int_rd(static_cast<float>(A) * inv_2out);
  int rem = A - i0 * D;
  if (rem < 0) {
    --i0;
    rem += D;
  } else if (rem >= D) {
    ++i0;
    rem -= D;
  }
  SrcCoord c;
  c.i0 = i0;
  c.w = static_cast<float>(rem) * inv_2out;
  return c;
}

// floor division for a possibly negative numerator, positive denominator
__device__ __forceinline__ int floor_div(int a, int d) {
  int q = a / d;
  if ((a % d != 0) && (a < 0)) --q;
  return q;
}

#endif  // __CUDACC__

}  // namespace mrx
