// sm_100a building blocks used by the tensor-core kernels: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (TMEM alloc / mma / commit / ld) PTX wrappers and the host-side tensor-map encoder.
#pragma once
#include <cuda.h>  // CUtensorMap (types only; the driver entry point is resolved at run time)

#include "common.cuh"

namespace rb {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier -----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug must surface as a trap (CUDA error), never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  long long t0 = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0xFFF) == 0) {
      long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000LL) {  // ~2 s at 2 GHz
        printf("raft_b200: mbarrier wait timed out (block %d,%d thread %d parity %u)\n", blockIdx.x, blockIdx.y,
               threadIdx.x, parity);
        __trap();
      }
    }
  }
}

// One lane of a CONVERGED warp.  Unlike `lane == 0`, ptxas knows that exactly one thread runs the guarded region, so the
// uniform-datapath instructions in it (UTCHMMA, UTMALDG, UTCBAR) are emitted directly instead of inside an
// elect / branch "waterfall" loop each (profiles/r01_notes.md: that loop was the k-iteration floor of the MMA warp).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// Whole-warp wait with ONE polling lane and a short back-off: 16 epilogue warps spinning with all lanes on the
// accumulator barrier for the length of an MMA loop compete with the producer / MMA threads for the barrier unit.
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity) {
  if ((threadIdx.x & 31) == 0) {
    uint32_t spins = 0;
    long long t0 = 0;
    while (!mbar_try_wait(bar, parity)) {
      __nanosleep(32);
      if ((++spins & 0x3FF) == 0) {
        long long now = clock64();
        if (t0 == 0) t0 = now;
        else if (now - t0 > 4000000000LL) {
          printf("raft_b200: mbarrier wait timed out (block %d warp %d parity %u)\n", blockIdx.x, threadIdx.x >> 5, parity);
          __trap();
        }
      }
    }
  }
  __syncwarp();
}

// ---- TMA ------------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---- tcgen05 ----------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle: rows are 128 B (64 fp16),
// 8-row core groups 1024 B apart (SBO); the tile base must be 1024-byte aligned.  Advancing by one
// UMMA_K (16 fp16 = 32 B) adds 2 to the 16-byte-granular start address.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);   // start address        bits [0,14)
  d |= (uint64_t)1 << 16;                       // LBO (unused for swizzled K-major) [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;             // SBO = 1024 B          bits [32,46)
  d |= (uint64_t)1 << 46;                       // descriptor version 1 (Blackwell)
  d |= (uint64_t)2 << 61;                       // layout type SWIZZLE_128B
  return d;
}
// Instruction descriptor, kind::f16: fp16 x fp16 -> fp32, both operands K-major, M=128.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int n) {
  return (1u << 4)                    // c_format = F32
         | (0u << 7) | (0u << 10)     // a_format = b_format = F16
         | ((uint32_t)(n >> 3) << 17) // N >> 3
         | ((uint32_t)(128 >> 4) << 24);  // M >> 4
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns: thread t of the warp gets row (lane base + t).
// The load is asynchronous: registers are valid only after tmem_ld_wait(), which names them as
// in/out operands so the compiler cannot hoist uses above the wait.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t* a, uint32_t* b) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                 "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                 "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]),
                 "+r"(b[8]), "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15])
               :
               : "memory");
}

// ---- host: tensor maps --------------------------------------------------------------------------------
// up to 4 dims (innermost first), zero fill for out-of-bounds boxes; kind selects element type and swizzle
enum { TMAP_F16_SW128 = 0, TMAP_F32_SW64 = 1, TMAP_F32_SW64_GATHER = 2 };  // GATHER: as SW64 but without L2 promotion (lookup v5)
int make_tmap(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
              const uint32_t* box, int kind, const uint32_t* elem_strides = nullptr);

}  // namespace tc

struct TileGeom {
  int bw_log2, bh_log2;  // box = 2^bh x 2^bw pixels, product 128
  int tiles_x, tiles_y;  // per image
  int n_tiles;           // cout tiles
  int m_tiles;           // B * tiles_x * tiles_y pixel tiles
  int total_tiles;       // work items: m_tiles * n_tiles
};

// per-thread cache of encoded tensor maps (conv_tc.cu)
int cached_tmap(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides,
                const uint32_t* box, int kind = tc::TMAP_F16_SW128, const uint32_t* elem_strides = nullptr);

}  // namespace rb

// ---- cluster building blocks (split-K pair of conv_tc.cu) -------------------------------------------------
namespace rb {
namespace tc {
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster_f32x2(uint32_t cluster_addr, float a, float b) {
  asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(cluster_addr), "f"(a), "f"(b) : "memory");
}
// wait whose acquire covers writes a peer CTA made to this CTA's shared memory before its release.cluster arrive
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0, spins = 0;
  long long t0 = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (ok) break;
    if ((++spins & 0xFFF) == 0) {
      long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000LL) {
        printf("raft_b200: cluster mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
}  // namespace tc
}  // namespace rb
