// Thin inline-PTX wrappers: mbarrier + 1-D TMA bulk copy (cp.async.bulk -> SASS UBLKCP),
// streaming loads/stores.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mdkm {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

// Make the barrier initialisation visible to the async (TMA) proxy.
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}

// 1-D bulk copy global -> shared, completion signalled on `bar` (complete_tx::bytes).
// dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// Address-form variants (shared-window addresses precomputed once per warp).
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d_a(uint32_t dst, const void* src_gmem, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src_gmem), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}

// One lane of the (converged) warp is elected; true in that lane only.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 r;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
  return r;
}

// Order this thread's generic-proxy shared-memory accesses before later async-proxy (TMA) ones.
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// Streaming (read-once) 128-bit load: read-only path, do not allocate in L1.
__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ uint32_t ldg_stream_u32(const void* p) {
  uint32_t r;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}

__device__ __forceinline__ uint2 ldg_stream_u64(const void* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}

// system-scope accesses for buffers that peer GPUs write / read over NVLink
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// Programmatic dependent launch: a kernel launched with the programmatic-stream-serialisation attribute
// may start while its predecessor in the stream still runs; it must not touch the predecessor's
// results before grid_dependency_wait() (a no-op for ordinary launches).
__device__ __forceinline__ void grid_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// gpu-scope release / acquire on a 32-bit flag (one CTA announces, the others of the grid wait)
__device__ __forceinline__ void st_release_gpu_u32(unsigned int* p, unsigned int v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_gpu_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// gpu-scope relaxed 32-bit accesses: union-find parents that other threads of the grid relink
__device__ __forceinline__ unsigned int ld_relaxed_gpu_u32(const void* p) {
  unsigned int v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_gpu_u32(void* p, unsigned int v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// 8-byte (value, flag) packets: one store / one load each, so a reader never sees one without the other
__device__ __forceinline__ void st_relaxed_sys_v2u32(void* p, unsigned int a, unsigned int b) {
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ uint2 ld_relaxed_sys_v2u32(const void* p) {
  uint2 v;
  asm volatile("ld.relaxed.sys.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}

// Decoupled look-back (single-pass exclusive scan over tiles that a ticket counter hands out in
// order, so every predecessor of a running tile is itself running or done).  Per-tile status
// word: flag in the two top bits, count below.
constexpr unsigned long long kStAggregate = 1ull << 62;  // value = items of this tile
constexpr unsigned long long kStPrefix = 2ull << 62;     // value = items up to and including this tile
constexpr unsigned long long kStValue = (1ull << 62) - 1ull;

__device__ __forceinline__ unsigned long long ld_status(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_status(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Items of all tiles before tile t (warp-collective; the tile's own aggregate has been published
// by the caller, except for tile 0).  Also publishes tile t's prefix.  Sums of up to 32 tiles must
// fit 32 bits.  Flag and value share one 64-bit status word, so no fence is
// involved: a word is either not there yet, an aggregate or a prefix.
__device__ __forceinline__ unsigned long long tile_lookback(unsigned long long* status, long long t, unsigned int agg,
                                                            int lane, unsigned int* fault) {
  unsigned long long excl = 0ull;
  const long long t0 = clock64();
  for (long long j = t - 1;; j -= 32) {
    const long long jj = j - lane;
    unsigned long long s;
    unsigned int first_pre, invalid;
    do {
      // bounded wait (about 4 s): every predecessor holds an earlier ticket, so it is running or done
      // and this never triggers; if it ever did, a flagged failure beats a hung GPU
      if (clock64() - t0 > (8ll << 30)) {
        if (lane == 0) atomicExch(fault, 1u);
        return 0ull;
      }
      s = jj >= 0 ? ld_status(status + jj) : kStPrefix;  // before tile 0: a prefix of zero items
      const unsigned int flag = (unsigned int)(s >> 62);
      const unsigned int pre = __ballot_sync(0xffffffffu, flag == 2u);
      first_pre = pre ? (unsigned int)__ffs(pre) - 1u : 32u;
      // every tile between t and the nearest prefix must have published its aggregate
      const unsigned int need = first_pre < 32u ? ((2u << first_pre) - 1u) : 0xffffffffu;
      invalid = __ballot_sync(0xffffffffu, flag == 0u) & need;
    } while (invalid);
    excl += __reduce_add_sync(0xffffffffu, (unsigned int)lane < first_pre ? (unsigned int)(s & kStValue) : 0u);
    if (first_pre < 32u) {
      excl += __shfl_sync(0xffffffffu, s, first_pre) & kStValue;
      break;
    }
  }
  if (lane == 0) st_status(status + t, kStPrefix | (excl + agg));
  return excl;
}

// warp-wide float min / max in one instruction (sm_100a: CREDUX.MIN/MAX.F32)
__device__ __forceinline__ float redux_min_f32(float v) {
  float r;
  asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ float redux_max_f32(float v) {
  float r;
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
  return r;
}

}  // namespace mdkm
