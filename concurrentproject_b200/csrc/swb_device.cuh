// swb_device.cuh -- thin primitives used by the wavefront engine.
//
// Every primitive has a device version (the product) and a host version that exists ONLY so
// tests/emu/engine_emu.cu can execute the very same engine body on CPU threads (one thread per
// lane, barriers for warp-synchronous points).  The shipped library never takes the host path:
// swb200.cu calls the engine exclusively from __global__ kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#if defined(__CUDA_ARCH__)
#define SWB_DEVICE_CODE 1
#else
#define SWB_DEVICE_CODE 0
#endif

#define SWB_HD __host__ __device__ __forceinline__

#if !SWB_DEVICE_CODE
#include <atomic>
#include <pthread.h>
#include <sched.h>
#endif

namespace swb {

// ---- packed 16-bit / 32-bit DPX arithmetic ---------------------------------------------------
// On sm_100a these compile to single SASS instructions: VIADD.16x2, VIADDMNMX.S16x2,
// VIMNMX3.S16x2.RELU, VIMNMX.S16x2, PRMT (checked with cuobjdump, see DESIGN.md).
SWB_HD uint32_t add16x2(uint32_t a, uint32_t b) {
#if SWB_DEVICE_CODE
  return __vadd2(a, b);
#else
  return ((a + b) & 0xFFFFu) | (((a >> 16) + (b >> 16)) << 16);
#endif
}
SWB_HD uint32_t addmax16x2(uint32_t a, uint32_t b, uint32_t c) { return __viaddmax_s16x2(a, b, c); }   // max(a+b, c)
SWB_HD uint32_t addmaxrelu16x2(uint32_t a, uint32_t b, uint32_t c) { return __viaddmax_s16x2_relu(a, b, c); }   // max(a+b, c, 0)
SWB_HD uint32_t max3relu16x2(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_s16x2_relu(a, b, c); }
SWB_HD uint32_t maxrelu16x2(uint32_t a, uint32_t b) { return __vimax_s16x2_relu(a, b); }                         // max(a, b, 0)
SWB_HD uint32_t max16x2(uint32_t a, uint32_t b) {
#if SWB_DEVICE_CODE
  return __vmaxs2(a, b);
#else
  const int al = (short)(a & 0xFFFFu), ah = (short)(a >> 16), bl = (short)(b & 0xFFFFu), bh = (short)(b >> 16);
  return ((uint32_t)(al > bl ? al : bl) & 0xFFFFu) | ((uint32_t)(ah > bh ? ah : bh) << 16);
#endif
}
SWB_HD uint32_t min16x2(uint32_t a, uint32_t b) {
#if SWB_DEVICE_CODE
  return __vmins2(a, b);
#else
  const int al = (short)(a & 0xFFFFu), ah = (short)(a >> 16), bl = (short)(b & 0xFFFFu), bh = (short)(b >> 16);
  return ((uint32_t)(al < bl ? al : bl) & 0xFFFFu) | ((uint32_t)(ah < bh ? ah : bh) << 16);
#endif
}
SWB_HD uint32_t max3_16x2(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_s16x2(a, b, c); }
SWB_HD int addmax32(int a, int b, int c) { return __viaddmax_s32(a, b, c); }
SWB_HD int addmaxrelu32(int a, int b, int c) { return __viaddmax_s32_relu(a, b, c); }
SWB_HD int max3relu32(int a, int b, int c) { return __vimax3_s32_relu(a, b, c); }
SWB_HD int max3_32(int a, int b, int c) { return __vimax3_s32(a, b, c); }

SWB_HD uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
#if SWB_DEVICE_CODE
  // not __byte_perm(): that intrinsic masks the selector with 0x7777 and loses the sign-replicate bit
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
#else
  // PTX prmt.b32 default mode: nibble k of sel picks byte (n&7) of {b,a}; bit 3 replicates its sign.
  uint64_t pool = ((uint64_t)b << 32) | a;
  uint32_t r = 0;
  for (int k = 0; k < 4; ++k) {
    uint32_t n = (sel >> (4 * k)) & 0xF;
    uint32_t byte = (uint32_t)(pool >> (8 * (n & 7))) & 0xFF;
    if (n & 8) byte = (byte & 0x80) ? 0xFF : 0x00;
    r |= byte << (8 * k);
  }
  return r;
#endif
}

// ---- global-memory flagged words ---------------------------------------------------------------
// Boundary entries are 8-byte {value, tag} words written with one store and polled with one load;
// a single aligned 8-byte access is indivisible, so no fence is needed between value and tag.
SWB_HD void st_entry(uint2* p, uint32_t value, uint32_t tag) {
#if SWB_DEVICE_CODE
  asm volatile("st.global.relaxed.sys.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(value), "r"(tag));
#else
  uint64_t v = ((uint64_t)tag << 32) | value;
  reinterpret_cast<std::atomic<uint64_t>*>(p)->store(v, std::memory_order_release);
#endif
}

SWB_HD uint2 ld_entry(const uint2* p) {
#if SWB_DEVICE_CODE
  uint2 r;
  asm volatile("ld.global.relaxed.sys.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
#else
  uint64_t v = reinterpret_cast<const std::atomic<uint64_t>*>(p)->load(std::memory_order_acquire);
  uint2 r; r.x = (uint32_t)v; r.y = (uint32_t)(v >> 32);
  return r;
#endif
}

// Read-only data fetched well before use: volatile so the compiler keeps the load where it is issued.
SWB_HD uint64_t ld_early_u64(const uint64_t* p) {
#if SWB_DEVICE_CODE
  uint64_t v;
  asm volatile("ld.global.nc.u64 %0, [%1];" : "=l"(v) : "l"(p));
  return v;
#else
  return *p;
#endif
}

SWB_HD void st_progress(unsigned long long* p, unsigned long long v) {
#if SWB_DEVICE_CODE
  asm volatile("st.global.relaxed.gpu.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
#else
  reinterpret_cast<std::atomic<unsigned long long>*>(p)->store(v, std::memory_order_release);
#endif
}

SWB_HD unsigned long long ld_progress(const unsigned long long* p) {
#if SWB_DEVICE_CODE
  unsigned long long v;
  asm volatile("ld.global.relaxed.gpu.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
#else
  return reinterpret_cast<const std::atomic<unsigned long long>*>(p)->load(std::memory_order_acquire);
#endif
}

SWB_HD int ld_flag(const int* p) {
#if SWB_DEVICE_CODE
  int v;
  asm volatile("ld.global.relaxed.gpu.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
#else
  return reinterpret_cast<const std::atomic<int>*>(p)->load(std::memory_order_acquire);
#endif
}

SWB_HD void atomic_max_i32(int* p, int v) {
#if SWB_DEVICE_CODE
  atomicMax(p, v);
#else
  auto* a = reinterpret_cast<std::atomic<int>*>(p);
  int cur = a->load();
  while (cur < v && !a->compare_exchange_weak(cur, v)) {}
#endif
}

SWB_HD void atomic_or_i32(int* p, int v) {
#if SWB_DEVICE_CODE
  atomicOr(p, v);
#else
  reinterpret_cast<std::atomic<int>*>(p)->fetch_or(v);
#endif
}

SWB_HD unsigned long long atomic_fetch_add_u64(unsigned long long* p, unsigned long long v) {
#if SWB_DEVICE_CODE
  return atomicAdd(p, v);
#else
  return reinterpret_cast<std::atomic<unsigned long long>*>(p)->fetch_add(v);
#endif
}

SWB_HD void spin_pause() {
#if SWB_DEVICE_CODE
  __nanosleep(20);
#else
  sched_yield();
#endif
}

// ---- bulk asynchronous copy (TMA, cp.async.bulk) + mbarrier: device only -------------------------
// Used by the TMA flavour of the pair engine (launch config 5) to stage a chunk of boundary entries from global
// memory (L2, or a peer GPU's stores that landed there) into shared memory.  The host emulation never takes this path.
#if SWB_DEVICE_CODE
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
#endif

// ---- warp context -------------------------------------------------------------------------------
#if SWB_DEVICE_CODE
struct WarpCtx {
  int lane;
  __device__ __forceinline__ uint32_t shfl(uint32_t v, int src) const { return __shfl_sync(0xffffffffu, v, src); }
  __device__ __forceinline__ void sync() const { __syncwarp(); }
  __device__ __forceinline__ int reduce_max(int v) const { return __reduce_max_sync(0xffffffffu, v); }
  __device__ __forceinline__ int any(int pred) const { return __any_sync(0xffffffffu, pred); }
  __device__ __forceinline__ int all(int pred) const { return __all_sync(0xffffffffu, pred); }
};
#else
// Host emulation: 32 threads per warp, a pthread barrier at every warp-synchronous point.
struct WarpShared {
  pthread_barrier_t bar;
  uint32_t slot[32];
};
struct WarpCtx {
  int lane;
  WarpShared* ws;
  uint32_t shfl(uint32_t v, int src) const {
    ws->slot[lane] = v;
    pthread_barrier_wait(&ws->bar);
    uint32_t r = ws->slot[src & 31];
    pthread_barrier_wait(&ws->bar);
    return r;
  }
  void sync() const { pthread_barrier_wait(&ws->bar); }
  int reduce_max(int v) const {
    ws->slot[lane] = (uint32_t)v;
    pthread_barrier_wait(&ws->bar);
    int r = (int)ws->slot[0];
    for (int k = 1; k < 32; ++k) r = (int)ws->slot[k] > r ? (int)ws->slot[k] : r;
    pthread_barrier_wait(&ws->bar);
    return r;
  }
  int all(int pred) const { return !any(!pred); }
  int any(int pred) const {
    ws->slot[lane] = (uint32_t)(pred != 0);
    pthread_barrier_wait(&ws->bar);
    int r = 0;
    for (int k = 0; k < 32; ++k) r |= (int)ws->slot[k];
    pthread_barrier_wait(&ws->bar);
    return r;
  }
};
#endif

}  // namespace swb
