// tcgen05 implicit-GEMM convolution / GEMM over split fp16 operands (the RB_MATH_TC back end).
//
// One CTA computes a 128-pixel x BLOCK_N-channel output tile.  The 128 pixels are a BH x BW box of
// one image, so for every filter tap the A operand is ONE TMA box load from the NHWC activation
// at a shifted coordinate -- out-of-image pixels are zero-filled by TMA, which is exactly TF 'SAME'
// zero padding for the stride-1 odd kernels of the update block (SURVEY A14).  Per (tap, 64-channel
// chunk) a pipeline stage holds A_hi, A_lo (128x64 fp16 each) and [B_hi ; B_lo] (2*BLOCK_N x 64),
// all 128-byte swizzled K-major.  Per 16-wide k-slice the MMA warp issues
//     D[:, 0:2N]  (+)= A_hi x [B_hi ; B_lo]^T      (N' = 2*BLOCK_N)
//     D[:, N:2N]   += A_lo x  B_hi^T
// so TMEM columns [0,N) hold hi*hi and [N,2N) hold the two cross terms (2^11-scaled); the
// epilogue forms hi*hi + 2^-11 * cross in fp32 and applies the fused epilogue of common.cuh.
// Warp roles: 0 = TMA producer, 1 = TMEM owner + MMA issuer, 2..17 = epilogue: warp w reads TMEM lane
// quarter (w % 4) and column group (w - 2) / 4 of 16 or 32 columns (profiles/r01: with 4 and then 8
// epilogue warps the dependent ALU chains of the epilogue took as long as the MMA loop).
// Programmatic dependent launch: the prologue (barrier init, TMEM allocation, descriptor prefetch) runs
// before griddepcontrol.wait, i.e. overlapped with the tail of the previous kernel in the stream.
#include <stdlib.h>
#include <unordered_map>
#include <string.h>

#include "tc_common.cuh"

namespace rb {
using namespace tc;

constexpr int kTileM = 128;
constexpr int kChunkK = 64;               // fp16 elements per 128-byte swizzled row
constexpr int kATileBytes = kTileM * 128;  // 16 KB
constexpr int kTcThreads = 576;            // 18 warps: TMA, MMA, 16 epilogue

// PERSISTENT kernel: each CTA walks tiles t = blockIdx.x, blockIdx.x + gridDim.x, ... (n-tile fastest, so CTAs that
// run side by side share the same activation tile in L2).  The accumulators are double-buffered in TMEM
// (2 x 2*BLOCK_N columns): the MMA warp starts the K loop of tile i+1 while the 16 epilogue warps drain tile i,
// and the smem ring / its mbarrier phases simply continue across tiles.  With one wave of tiles (the update block
// at batch 1) this degenerates to one tile per CTA; with many tiles (batched runs, encoder layers, the 3025-tile
// correlation GEMM) the epilogue disappears behind the next tile's MMA loop.
template <int BLOCK_N>
struct TcCfg {
  static constexpr int kBTileBytes = BLOCK_N * 128;
  static constexpr int kStageBytes = 2 * kATileBytes + 2 * kBTileBytes;
  static constexpr int kStages = (200 * 1024) / kStageBytes > 6 ? 6 : (200 * 1024) / kStageBytes;
  static constexpr int kAccCols = 2 * BLOCK_N;  // hi*hi | cross terms
  // two accumulator buffers; tiles of >= 32 columns take all 512 columns: a CTA that owns a single tile (batch 1) parks
  // the fp32 operands of the gate epilogues behind its one live buffer (Stash, common.cuh) -- up to 3 x BLOCK_N columns
  // 16-wide tiles keep room for a second accumulator per buffer (K summed in two halves, see split_k below)
  static constexpr int kBufCols = BLOCK_N == 16 ? 2 * kAccCols : kAccCols;
  static constexpr int kTmemCols = BLOCK_N == 16 ? 128 : 512;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/ + 1024 /*split-K partials*/;
  static constexpr int kColsPerWarp = BLOCK_N >= 96 ? 32 : 16;
  static constexpr int kGroups = BLOCK_N / kColsPerWarp;  // 128:4  96:3  64:4  32:2  16:1 column groups of epilogue warps
};


// EXTRAS: phase timestamps (p.dbg) and fused instance-norm statistics (p.stat_part) -- a separate instantiation, so that
// the kernel the update block runs stays below the 96-register cap of a 576-thread CTA without spills.
template <int BLOCK_N, bool EXTRAS>
__global__ void __launch_bounds__(kTcThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
               const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
               const ConvParams p, const TileGeom g, const int STAGES) {
  using Cfg = TcCfg<BLOCK_N>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::kStageBytes);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;   // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  uint64_t* red_bar = tmem_empty_bar + 3;  // split-K: the peer's partial sums have arrived (128 lane arrivals)
  float2* red_buf = reinterpret_cast<float2*>(smem + STAGES * Cfg::kStageBytes + 256);  // [128 pixels] channels 0, 1

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  long long* dbg = (EXTRAS && p.dbg) ? p.dbg + (size_t)blockIdx.x * 8 : nullptr;
  const bool wide = epilogue_wide_ok(p);
  if (dbg && threadIdx.x == 0) dbg[0] = gtime_ns();
  // Split-K (p.split_k, 16-wide tiles with <= 2 real channels: the flow head's last conv, update.cu).  The sum over K is
  // ALWAYS formed as (first half of the channel chunks) + (second half), each half in its own accumulator, so that the
  // result does not depend on how it is executed:
  //  * p.split_cluster = 1 (one wave of CTA pairs, batch 1): clusters of two CTAs share one pixel tile, CTA r multiplies
  //    half r; CTA 1 hands its partial sums to CTA 0 through distributed shared memory, CTA 0 runs the epilogue on r0 + r1;
  //  * else one CTA runs both halves back to back into two TMEM accumulators and its epilogue adds them the same way.
  const bool halves = BLOCK_N == 16 && p.split_k;
  const bool splitk = halves && p.split_cluster;
  const int chunks = splitk ? conv_chunks(p) / 2 : conv_chunks(p);
  const int taps = p.kh * p.kw;
  const int kiters = taps * chunks;
  const int tiles_per_img = g.tiles_x * g.tiles_y;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA_hi); prefetch_tmap(&tmA_lo); prefetch_tmap(&tmB_hi); prefetch_tmap(&tmB_lo);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full_bar[i], 1); mbar_init(&tmem_empty_bar[i], Cfg::kGroups * 4); }
    mbar_init(red_bar, 128);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  tc_fence_before();
  __syncthreads();
  if (splitk) cluster_sync_all();  // the peer's barriers must be initialised before anything of ours can reach them
  tc_fence_after();
  // warp-wide OR of identical values: lands in a UNIFORM register, so that ptxas does not wrap every tcgen05.mma of the
  // single issuing lane in an elect / R2UR.BROADCAST "waterfall" loop (that was ~50 cycles per MMA, 8 MMAs per k-iteration)
  const uint32_t tmem_base = __reduce_or_sync(0xffffffffu, *tmem_slot);
  const int krank = splitk ? (int)cluster_ctarank() : 0;
  const int first = splitk ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;      // first work item of this CTA (pair)
  const int stride = splitk ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  if (dbg && threadIdx.x == 0) dbg[1] = gtime_ns();
  // Programmatic dependent launch: this kernel may have been started while its predecessor is still running.  Everything
  // up to here (barriers, TMEM, tensor-map prefetch) and the WEIGHT tiles of the first ring stages are independent of
  // it; `griddepcontrol.wait` (no-op without the launch attribute) is executed by the producer before its first
  // activation load and by every epilogue warp before its first global access.  The MMA warp touches no global memory.

  if (warp == 0) {
    if (elect_one()) {
      const int ph = conv_pad_y(p), pw = conv_pad_x(p), csx = conv_sx(p), csy = conv_sy(p);
      int s = 0;          // ring slot and its phase; both continue across tiles.  No integer division in this loop:
      uint32_t phase = 0;  // the k-iteration -> (chunk, kx, ky) mapping is advanced incrementally.
      bool waited = false;
      for (int tile = first; tile < g.total_tiles; tile += stride) {
        const int mt = tile / g.n_tiles, nt = tile - mt * g.n_tiles;
        const int b = mt / tiles_per_img, trem = mt - b * tiles_per_img;
        const int ty = trem / g.tiles_x, tx = trem - ty * g.tiles_x;
        const int y0 = ty << g.bh_log2, x0 = tx << g.bw_log2, n0 = nt * BLOCK_N;
        const int xs = x0 * csx - pw, ys = y0 * csy - ph;  // input coordinates of tap (0, 0) of the tile's first pixel
        const int wb = p.w_per_batch ? min(b, p.B - 1) : 0;
        // K order: channel chunk outermost, then kx, then ky.  The order is fixed, whatever the tile geometry or the
        // number of tiles per CTA, so a batched run equals the per-sample runs bit for bit.
        struct KIter {
          int cki, kx, ky, ck;
        };
        auto k_next = [&](KIter& k) {
          if (++k.ky == p.kh) {
            k.ky = 0;
            if (++k.kx == p.kw) { k.kx = 0; k.ck = conv_chunk(p, ++k.cki); }
          }
        };
        auto load_a = [&](const KIter& k, int slot) {
          uint8_t* st = smem + slot * Cfg::kStageBytes;
          const int c0 = p.in_choff + k.ck * kChunkK;
          tma_load_4d(&tmA_hi, &full_bar[slot], st, c0, xs + k.kx, ys + k.ky, b);
          tma_load_4d(&tmA_lo, &full_bar[slot], st + kATileBytes, c0, xs + k.kx, ys + k.ky, b);
        };
        auto load_b = [&](const KIter& k, int slot) {
          uint8_t* st = smem + slot * Cfg::kStageBytes;
          const int kcol = (k.ky * p.kw + k.kx) * p.cin_pad + k.ck * kChunkK;
          tma_load_3d(&tmB_hi, &full_bar[slot], st + 2 * kATileBytes, kcol, n0, wb);
          tma_load_3d(&tmB_lo, &full_bar[slot], st + 2 * kATileBytes + Cfg::kBTileBytes, kcol, n0, wb);
        };
        KIter k = {krank * chunks, 0, 0, conv_chunk(p, krank * chunks)};
        int it0 = 0;
        if (!waited) {
          // first tile of the kernel: weight tiles of the first ring stages, then wait for the predecessor kernel, then
          // the activation tiles of the same stages (the ring is empty here: slots 0.., phase 0)
          // (not when the B operand is itself an activation produced by an earlier kernel: corr build, w_per_batch)
          const int pre = p.w_per_batch ? 0 : (kiters < STAGES ? kiters : STAGES);
          KIter kb = k;
          for (int it = 0; it < pre; ++it) {
            mbar_arrive_expect_tx(&full_bar[it], Cfg::kStageBytes);
            load_b(kb, it);
            k_next(kb);
          }
          asm volatile("griddepcontrol.wait;" ::: "memory");
          if (dbg) dbg[2] = gtime_ns();
          for (int it = 0; it < pre; ++it) {
            load_a(k, s);
            k_next(k);
            if (++s == STAGES) { s = 0; phase ^= 1; }
          }
          it0 = pre;
          waited = true;
        }
        for (int it = it0; it < kiters; ++it) {
          mbar_wait(&empty_bar[s], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[s], Cfg::kStageBytes);
          load_a(k, s);
          load_b(k, s);
          k_next(k);
          if (++s == STAGES) { s = 0; phase ^= 1; }
        }
      }
    }
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_2n = umma_idesc_f16(2 * BLOCK_N);
      constexpr uint32_t idesc_n = umma_idesc_f16(BLOCK_N);
      int s = 0, li = 0;
      uint32_t phase = 0;
      for (int tile = first; tile < g.total_tiles; tile += stride, ++li) {
        const int ab = li & 1;
        mbar_wait(&tmem_empty_bar[ab], ((li >> 1) & 1) ^ 1);  // epilogue has drained this accumulator buffer
        tc_fence_after();
        uint32_t acc = tmem_base + ab * Cfg::kBufCols;
        const int it_half = (halves && !splitk) ? kiters / 2 : -1;  // first k-iteration of the second accumulator
        for (int it = 0; it < kiters; ++it) {
          if constexpr (BLOCK_N == 16) {
            if (it == it_half) acc += Cfg::kAccCols;
          }
          mbar_wait(&full_bar[s], phase);
          tc_fence_after();
          if (dbg && li == 0 && it == 0) dbg[3] = gtime_ns();
          const uint32_t st = smem_u32(smem + s * Cfg::kStageBytes);
          const uint64_t a_hi = umma_desc_sw128(st);
          const uint64_t a_lo = umma_desc_sw128(st + kATileBytes);
          const uint64_t b_all = umma_desc_sw128(st + 2 * kATileBytes);  // [B_hi ; B_lo], 2N rows
#pragma unroll
          for (int k = 0; k < kChunkK / 16; ++k) {
            const uint64_t koff = (uint64_t)(k * 2);  // 32 bytes per k-slice, in 16-byte units
            umma_f16(acc, a_hi + koff, b_all + koff, idesc_2n, (BLOCK_N == 16 ? ((it != 0 && it != it_half) || k != 0) : (it | k) != 0));
            umma_f16(acc + BLOCK_N, a_lo + koff, b_all + koff, idesc_n, 1u);
          }
          umma_commit(&empty_bar[s]);  // frees the smem stage when these MMAs retire
          if (++s == STAGES) { s = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full_bar[ab]);
        if (dbg && li == 0) dbg[4] = gtime_ns();
      }
    }
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  } else {
    // ---- epilogue: warps 2..17 -- lane quarter (warp % 4), column group (warp - 2) / 4 ----
    const int q = warp & 3;
    const int grp = (warp - 2) >> 2;
    const int r = q * 32 + lane;  // tile row = pixel index inside the box
    if (grp >= Cfg::kGroups) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (grp < Cfg::kGroups) {
      asm volatile("griddepcontrol.wait;" ::: "memory");  // addend / z / h reads and all stores come after the predecessor
      int li = 0;
      // ---- operand stash (see common.cuh): single-tile CTAs of the GRU gate convs, while the MMA loop runs ----
      uint32_t stash_row = 0;
      if constexpr (!EXTRAS && BLOCK_N >= 32) {
        const int nops = p.epi == EPI_Q ? 3 : 2;
        if (p.stash && wide && (p.epi == EPI_ZR || p.epi == EPI_Q) && g.total_tiles <= (int)gridDim.x &&
            Cfg::kAccCols + nops * BLOCK_N <= Cfg::kTmemCols && first < g.total_tiles) {
          const int mq = first / g.n_tiles, nt = first - mq * g.n_tiles;
          const int b = mq / tiles_per_img, trem = mq - b * tiles_per_img;
          const int ty = trem / g.tiles_x, tx = trem - ty * g.tiles_x;
          const int py = (ty << g.bh_log2) + (r >> g.bw_log2), px = (tx << g.bw_log2) + (r & ((1 << g.bw_log2) - 1));
          const bool valid = (py < p.h) && (px < p.w) && (mq < g.m_tiles);
          const int pix = (b * p.h + py) * p.w + px, n0 = nt * BLOCK_N;
          stash_row = tmem_base + ((uint32_t)(q * 32) << 16) + Cfg::kAccCols;
#pragma unroll 1
          for (int cc = 0; cc < Cfg::kColsPerWarp; cc += 16) {
            const int c = grp * Cfg::kColsPerWarp + cc;
            if (n0 + c >= p.cout) break;  // warp-uniform
            float t[16];
            auto fetch = [&](const float* src) {
              if (valid) { ld256_nc(src, t); ld256_nc(src + 8, t + 8); }
              else {
#pragma unroll
                for (int i = 0; i < 16; ++i) t[i] = 0.f;
              }
            };
            if (p.addend) { fetch(p.addend + (size_t)pix * p.cout + n0 + c); tmem_st16(stash_row + c, t); }
            if (p.epi == EPI_ZR) {
              if (n0 + c >= p.hidden) {  // r half: h (model_utils.py:144,153)
                fetch(p.f1 + (size_t)pix * p.hidden + (n0 + c - p.hidden));
                tmem_st16(stash_row + BLOCK_N + c, t);
              }
            } else {  // EPI_Q: z and h (model_utils.py:147,155)
              fetch(p.f0 + (size_t)pix * p.hidden + n0 + c);
              tmem_st16(stash_row + BLOCK_N + c, t);
              fetch(p.f1 + (size_t)pix * p.hidden + n0 + c);
              tmem_st16(stash_row + 2 * BLOCK_N + c, t);
            }
          }
          tmem_st_wait();
        }
      }
      for (int tile = first; tile < g.total_tiles; tile += stride, ++li) {
        const int mt = tile / g.n_tiles, nt = tile - mt * g.n_tiles;
        const int b = mt / tiles_per_img, trem = mt - b * tiles_per_img;
        const int ty = trem / g.tiles_x, tx = trem - ty * g.tiles_x;
        const int y0 = ty << g.bh_log2, x0 = tx << g.bw_log2, n0 = nt * BLOCK_N;
        const int py = y0 + (r >> g.bw_log2), px = x0 + (r & ((1 << g.bw_log2) - 1));
        const bool valid = (py < p.h) && (px < p.w) && (mt < g.m_tiles);
        const int pix = (b * p.h + py) * p.w + px;
        const int ab = li & 1;
        mbar_wait_warp(&tmem_full_bar[ab], (li >> 1) & 1);
        tc_fence_after();
        if (li == 0) {
          asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
          if (dbg && warp == 2 && lane == 0) dbg[5] = gtime_ns();
        }
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + ab * Cfg::kBufCols;
#pragma unroll 1
        for (int cc = 0; cc < Cfg::kColsPerWarp; cc += 16) {
          const int c = grp * Cfg::kColsPerWarp + cc;
          if (n0 + c >= p.cout) break;  // warp-uniform
          uint32_t d0[16], d1[16];
          tmem_ld16(trow + c, d0);
          tmem_ld16(trow + BLOCK_N + c, d1);
          tmem_ld_wait(d0, d1);
          float v[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(d0[i]) + __uint_as_float(d1[i]) * kLoInv;
          bool store = valid;
          if constexpr (BLOCK_N == 16) {
            if (halves && !splitk) {  // second accumulator of the same CTA
              tmem_ld16(trow + Cfg::kAccCols + c, d0);
              tmem_ld16(trow + Cfg::kAccCols + BLOCK_N + c, d1);
              tmem_ld_wait(d0, d1);
              v[0] += __uint_as_float(d0[0]) + __uint_as_float(d1[0]) * kLoInv;
              v[1] += __uint_as_float(d0[1]) + __uint_as_float(d1[1]) * kLoInv;
            }
            if (splitk) {
              if (krank != 0) {  // partial sums of channels 0, 1 -> CTA 0 of the cluster; nothing else to do here
                st_cluster_f32x2(mapa_u32(smem_u32(red_buf + r), 0), v[0], v[1]);
                mbar_arrive_remote(mapa_u32(smem_u32(red_bar), 0));
                store = false;
              } else {
                mbar_wait_cluster(red_bar, 0);
                const float2 t = red_buf[r];
                v[0] += t.x;
                v[1] += t.y;
              }
            }
          }
          if (store || stash_row != 0) {  // with a stash the TMEM reads inside are warp-collective: all lanes go
            if (wide) {
              epilogue_wide16(p, pix, n0 + c, v, Stash{stash_row, BLOCK_N, c}, valid);
            } else {
              epilogue_store<8>(p, pix, n0 + c, v);
              epilogue_store<8>(p, pix, n0 + c + 8, v + 8);
            }
          }
          if (EXTRAS && p.stat_part) {  // instance-norm statistics of the values just stored (v was finalised in place; host: wide only)
            if (!valid) {
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] = 0.f;
            }
            float s1, s2;
            int ch;
            warp_stats16(v, s1, s2, ch);
            if ((lane & 1) == 0 && mt < g.m_tiles) {
              double* dst = p.stat_part + ((size_t)(b * p.stat_strips + trem * 4 + q) * 2) * p.cout + n0 + c + ch;
              dst[0] = (double)s1;
              dst[p.cout] = (double)s2;
            }
          }
        }
        // this warp no longer needs the accumulator buffer: hand it back to the MMA warp
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&tmem_empty_bar[ab])) : "memory");
        }
      }
    }
  }
  if (dbg && warp == 2 && lane == 0) dbg[6] = gtime_ns();
  tc_fence_before();
  __syncthreads();
  // Split-K: CTA 0 cannot exit before CTA 1's partial sums have landed in its shared memory -- it waited for them
  // (mbarrier, release.cluster / acquire.cluster) -- so no closing cluster barrier is needed.  compute-sanitizer's racecheck
  // cannot see that ("block that might have already exited"); p.split_close adds the barrier it wants (0 hazards with it,
  // +1 us per update step: profiles/r02_notes.md).
  if (splitk && p.split_close) cluster_sync_all();
  if (dbg && threadIdx.x == 0) dbg[7] = gtime_ns();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ---- host side -------------------------------------------------------------------------------------
namespace tc {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

int make_tmap(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
              const uint32_t* box, int kind, const uint32_t* elem_strides) {
  EncodeTiledFn fn = encode_fn();
  RB_REQUIRE(fn, RB_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t gdim[5];
  cuuint64_t gstr[5];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; es[i] = elem_strides ? elem_strides[i] : 1; }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  const CUtensorMapDataType dt = kind == TMAP_F16_SW128 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  const CUtensorMapSwizzle sw = kind == TMAP_F16_SW128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  // L2 promotion: 256-byte requests suit the dense 128-byte operand rows of the GEMM tiles; the lookup's 64-byte patch
  // rows are a gather (r01: 1.86x the algorithmic DRAM bytes) -> none.
  const CUtensorMapL2promotion promo =
      kind == TMAP_F32_SW64_GATHER ? CU_TENSOR_MAP_L2_PROMOTION_NONE : CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
  CUresult r = fn(out, dt, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RB_REQUIRE(r == CUDA_SUCCESS, RB_ERR_CUDA,
             "cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu,%llu,%llu,%llu] box [%u,%u,%u,%u]", (int)r, rank,
             (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
             (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0), box[0],
             rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
  return RB_OK;
}
}  // namespace tc

// Tensor maps depend only on (pointer, geometry); cache them per thread so steady-state launches
// (and CUDA-graph capture, which bakes kernel parameters) pay nothing for the encode.
struct TmapKey {
  const void* base;
  uint64_t kind;
  uint64_t d[4];
  uint64_t s[4];
  uint32_t b[4];
  uint32_t e[4];
  bool operator==(const TmapKey& o) const { return memcmp(this, &o, sizeof(TmapKey)) == 0; }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    const uint64_t* w = reinterpret_cast<const uint64_t*>(&k);
    size_t h = 1469598103934665603ull;
    for (size_t i = 0; i < sizeof(TmapKey) / 8; ++i) h = (h ^ w[i]) * 1099511628211ull;
    return h;
  }
};

int cached_tmap(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides,
                const uint32_t* box, int kind, const uint32_t* elem_strides) {
  static thread_local std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> cache;
  TmapKey k;
  memset(&k, 0, sizeof(k));
  k.base = base;
  k.kind = (uint64_t)kind;
  for (int i = 0; i < rank; ++i) {
    k.d[i] = dims[i]; k.s[i] = (i + 1 < rank) ? strides[i] : 0; k.b[i] = box[i]; k.e[i] = elem_strides ? elem_strides[i] : 1;
  }
  auto it = cache.find(k);
  if (it != cache.end()) { *out = it->second; return RB_OK; }
  int rc = make_tmap(out, base, rank, dims, strides, box, kind, elem_strides);
  if (rc) return rc;
  if (cache.size() > 4096) cache.clear();
  cache.emplace(k, *out);
  return RB_OK;
}

static TileGeom choose_geom(int h, int w) {
  TileGeom best{};
  long best_tiles = -1;
  for (int bwl = 7; bwl >= 3; --bwl) {
    int bw = 1 << bwl, bh = kTileM >> bwl;
    if (bw > w && bwl > 3) continue;  // keep the box inside the row when possible
    long tiles = (long)((w + bw - 1) / bw) * ((h + bh - 1) / bh);
    if (best_tiles < 0 || tiles < best_tiles) {
      best_tiles = tiles;
      best.bw_log2 = bwl; best.bh_log2 = 7 - bwl;
      best.tiles_x = (w + bw - 1) / bw; best.tiles_y = (h + bh - 1) / bh;
    }
  }
  return best;
}

// Pixel tiles per image of the tensor-core conv (strip count of the fused instance-norm statistics = 4x this).
int conv_tc_tiles_per_image(int h, int w) {
  const TileGeom g = choose_geom(h, w);
  return g.tiles_x * g.tiles_y;
}
// The conv can produce the statistics itself: tensor-core back end, 16-channel epilogue (see epilogue_wide_ok()).
bool conv_tc_fused_stats_ok(const ConvParams& p) {
  static const bool off = getenv("RAFT_B200_NO_FUSED_STATS") != nullptr;  // A/B knob
  auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 31) == 0; };
  return !off && math_mode() == RB_MATH_TC && p.epi == EPI_F32 && (p.cout & 15) == 0 && al(p.bias) && al(p.addend) && al(p.f0) &&
         p.cin_pad % kChunkK == 0;
}

// cycles per 16-wide k-slice: max(tensor math, shared-memory operand reads), see DESIGN.md
static int slice_cycles(int n) {
  int math = n + n / 2;
  int smem = 64 + (3 * n) / 4;
  return math > smem ? math : smem;
}

static int choose_block_n(int cout, long m_tiles, int ctas = 148) {  // ctas: persistent CTAs the launch may use (cta_limit)
  if (cout <= 16) return 16;
  const int cand[4] = {128, 96, 64, 32};
  int best = 128;
  long best_cost = -1;
  for (int i = 0; i < 4; ++i) {
    int n = cand[i];
    long tiles = m_tiles * ((cout + n - 1) / n);
    long waves = (tiles + ctas - 1) / ctas;
    long cost = waves * slice_cycles(n);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = n; }
  }
  return best;
}

template <int BLOCK_N>
static int launch_cfg(const ConvParams& p_in, TileGeom g, const CUtensorMap* maps, cudaStream_t s) {
  using Cfg = TcCfg<BLOCK_N>;
  static PerDeviceOnce attr_set;
  int dev = 0, rc_dev;
  if ((rc_dev = current_device(&dev))) return rc_dev;
  if (!attr_set.test(dev)) {
    RB_CHECK_CUDA(cudaFuncSetAttribute(conv_tc_kernel<BLOCK_N, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    RB_CHECK_CUDA(cudaFuncSetAttribute(conv_tc_kernel<BLOCK_N, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set.set(dev);
  }
  const int num_sms = device_sm_count(dev);
  ConvParams p = p_in;
  g.n_tiles = (p.cout + BLOCK_N - 1) / BLOCK_N;
  g.m_tiles = p.B * g.tiles_x * g.tiles_y;
  g.total_tiles = g.m_tiles * g.n_tiles;
  // split-K: only when every pixel tile gets its own CTA pair in one wave (batch 1), else the plain persistent grid
  if (p.split_k && !(BLOCK_N == 16 && p.cout <= 2 && p.epi == EPI_DELTA && !p.w_per_batch && conv_chunks(p) % 2 == 0))
    p.split_k = 0;
  static const bool no_cluster = getenv("RAFT_B200_NO_SPLITK_CLUSTER") != nullptr;  // test knob: same sums on one CTA
  static const bool close_barrier = getenv("RAFT_B200_SPLITK_CLOSING_BARRIER") != nullptr;  // for compute-sanitizer runs
  p.split_close = close_barrier ? 1 : 0;
  p.split_cluster = (p.split_k && 2 * g.total_tiles <= num_sms && p.cta_limit <= 0 && !no_cluster) ? 1 : 0;
  const bool cluster2 = p.split_cluster;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  int units = cluster2 ? num_sms / 2 : num_sms;  // persistent: at most one CTA (pair) per SM (pair)
  if (!cluster2 && p.cta_limit > 0 && p.cta_limit < units) units = p.cta_limit;  // leave SMs to a concurrent conv (update.cu)
  cfg.gridDim = dim3((g.total_tiles < units ? g.total_tiles : units) * (cluster2 ? 2 : 1));
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster2 ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  // Programmatic dependent launch (RAFT_B200_NO_PDL=1 turns it off): the dependent conv's prologue and its first
  // weight tiles overlap the tail of this one.  Same-box A/B after the issue-loop fixes: 190 -> 175 us per update step.
  static const int pdl = getenv("RAFT_B200_NO_PDL") ? 0 : 1;
  cfg.numAttrs = 1 + pdl;
  const int stages = Cfg::kStages;
  if (p.dbg || p.stat_part)
    RB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<BLOCK_N, true>, maps[0], maps[1], maps[2], maps[3], p, g, stages));
  else
    RB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<BLOCK_N, false>, maps[0], maps[1], maps[2], maps[3], p, g, stages));
  RB_CHECK_LAUNCH("conv_tc_kernel");
  return RB_OK;
}

int launch_conv_tc(const ConvParams& p, cudaStream_t s) {
  RB_REQUIRE(p.cin_pad % kChunkK == 0 && p.in_stride % 8 == 0 && p.in_choff % 8 == 0, RB_ERR_BAD_SHAPE,
             "conv_tc: channel padding (cin_pad=%d stride=%d off=%d)", p.cin_pad, p.in_stride, p.in_choff);
  const TileGeom g = choose_geom(p.h, p.w);
  const long m_tiles = (long)p.B * g.tiles_x * g.tiles_y;
  const int bn = choose_block_n(p.cout, m_tiles, p.cta_limit > 0 && p.cta_limit < 148 ? p.cta_limit : 148);
  CUtensorMap maps[4];
  {
    // the input view (common.cuh): strided convs traverse it with TMA element strides -- a box of bw*sx x bh*sy input
    // pixels delivers every sx-th / sy-th one, i.e. the bw x bh taps of the output tile
    const int iw = conv_in_w(p), ih = conv_in_h(p), sx = conv_sx(p), sy = conv_sy(p);
    const uint64_t rowpitch = (uint64_t)conv_rowpitch(p);
    RB_REQUIRE(sx <= 2 && sy <= 2 && rowpitch % 8 == 0, RB_ERR_BAD_SHAPE, "conv_tc: stride (%d,%d) / row pitch %llu", sx, sy,
               (unsigned long long)rowpitch);
    uint64_t dims[4] = {(uint64_t)(p.in_cext > 0 ? p.in_cext : p.in_stride), (uint64_t)iw, (uint64_t)ih, (uint64_t)p.B};
    uint64_t str[3] = {(uint64_t)p.in_stride * 2, rowpitch * 2, rowpitch * 2 * ih};
    uint32_t box[4] = {(uint32_t)kChunkK, (1u << g.bw_log2) * sx, (1u << g.bh_log2) * sy, 1};
    uint32_t es[4] = {1, (uint32_t)sx, (uint32_t)sy, 1};
    int rc;
    if ((rc = cached_tmap(&maps[0], p.in_hi, 4, dims, str, box, tc::TMAP_F16_SW128, es))) return rc;
    if ((rc = cached_tmap(&maps[1], p.in_lo, 4, dims, str, box, tc::TMAP_F16_SW128, es))) return rc;
  }
  {
    const uint64_t ktot = (uint64_t)p.kh * p.kw * p.cin_pad;
    uint64_t dims[3] = {ktot, (uint64_t)p.cout_pad, (uint64_t)(p.w_per_batch ? p.B : 1)};
    uint64_t str[2] = {ktot * 2, ktot * 2 * p.cout_pad};
    uint32_t box[3] = {(uint32_t)kChunkK, (uint32_t)bn, 1};
    int rc;
    if ((rc = cached_tmap(&maps[2], p.w_hi, 3, dims, str, box))) return rc;
    if ((rc = cached_tmap(&maps[3], p.w_lo, 3, dims, str, box))) return rc;
  }
  switch (bn) {
    case 16: return launch_cfg<16>(p, g, maps, s);
    case 32: return launch_cfg<32>(p, g, maps, s);
    case 64: return launch_cfg<64>(p, g, maps, s);
    case 96: return launch_cfg<96>(p, g, maps, s);
    default: return launch_cfg<128>(p, g, maps, s);
  }
}

}  // namespace rb
