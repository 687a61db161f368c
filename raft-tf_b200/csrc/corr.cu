// A1 (correlation volume + pyramid), A2/A3 (pyramid lookup), A4 (coords grid).
// Reference: networks/model_utils.py:199-249, networks/utils.py:4-103.
#include <stdlib.h>
#include <string.h>

#include "tc_common.cuh"

namespace rb {

// ---------------------------------------------------------------------------------------------
// A4  coords_grid  (utils.py:4-11)
// ---------------------------------------------------------------------------------------------
__global__ void coords_grid_kernel(float2* __restrict__ coords, int B, int h, int w) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int n = B * h * w;
  if (i >= n) return;
  int x = i % w, y = (i / w) % h;
  coords[i] = make_float2((float)x, (float)y);
}

// ---------------------------------------------------------------------------------------------
// A1  SIMT fp32 correlation GEMM: vol[b, n, m] = <f1[b,n,:], f2[b,m,:]> / sqrt(C)
//     (model_utils.py:206-215).  64x64 tile, 16-deep k slices, 4x4 micro-tile per thread.
//     Bring-up / cross-check back end (RB_MATH_SIMT); the tcgen05 build lives in gemm_tc.cu.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) corr_gemm_simt_kernel(const float* __restrict__ f1,
                                                             const float* __restrict__ f2,
                                                             float* __restrict__ vol, int N, int C,
                                                             float inv_sqrt_c_is_unused) {
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const int b = blockIdx.z;
  const float* A = f1 + (size_t)b * N * C;
  const float* Bm = f2 + (size_t)b * N * C;
  float* out = vol + (size_t)b * N * N;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < C; k0 += 16) {
    {
      int r = tid / 4, kq = (tid % 4) * 4;
      float4 va = make_float4(0, 0, 0, 0), vb = va;
      if (m0 + r < N) va = *reinterpret_cast<const float4*>(A + (size_t)(m0 + r) * C + k0 + kq);
      if (n0 + r < N) vb = *reinterpret_cast<const float4*>(Bm + (size_t)(n0 + r) * C + k0 + kq);
      As[kq + 0][r] = va.x; As[kq + 1][r] = va.y; As[kq + 2][r] = va.z; As[kq + 3][r] = va.w;
      Bs[kq + 0][r] = vb.x; Bs[kq + 1][r] = vb.y; Bs[kq + 2][r] = vb.z; Bs[kq + 3][r] = vb.w;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float a[4], bb[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; bb[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
  const float sq = sqrtf((float)C);
  for (int i = 0; i < 4; ++i) {
    int m = m0 + ty * 4 + i;
    if (m >= N) continue;
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n < N) out[(size_t)m * N + n] = acc[i][j] / sq;  // divide AFTER the matmul (:213)
    }
  }
}

// 2x2 average pooling, stride 2, VALID (floor) -- tensorpack AvgPooling (model_utils.py:217-219).
__global__ void avgpool2_kernel(const float* __restrict__ src, float* __restrict__ dst, size_t rows,
                                int hs, int ws, int hd, int wd) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t total = rows * hd * wd;
  if (i >= total) return;
  int x = i % wd;
  int y = (i / wd) % hd;
  size_t r = i / ((size_t)wd * hd);
  const float* s = src + r * hs * ws + (size_t)(2 * y) * ws + 2 * x;
  dst[i] = (s[0] + s[1] + s[ws] + s[ws + 1]) * 0.25f;
}

// ---------------------------------------------------------------------------------------------
// A2/A3  pyramid lookup (model_utils.py:224-249 + utils.py:39-103).
//
// A block handles PB = 8 query pixels x 4 levels = 32 "units"; thread = (unit, window row j).
//   phase 0  thread u computes the origin of unit u's footprint and -- when the level's rows are 16-byte
//            aligned -- issues ONE TMA box load (16 columns x (2r+3) rows of fp32, 64-byte swizzle) for it:
//            the (2r+1)^2 taps share one fractional offset, so their bilinear footprints tile a (2r+2)^2 patch
//            (+1 row/col of slack for the fp32 rounding of cx+dx, +<=3 columns of alignment).  Out-of-image parts
//            of the box are zero-filled and never indexed (tap indices are clamped like the reference's).
//            Levels whose width is not a multiple of 4 are staged with plain loads instead.
//   phase 1  thread j of a unit computes the x-side of window column i=j (clamped x0/x1 relative to the staged
//            columns, qx = x1c - x and 1 - qx) into a shared table and keeps the y-side of its own row j in
//            registers: the separable index math is done once per row / column instead of once per tap.
//   phase 2  each thread walks the (2r+1) taps of its row with the reference's exact arithmetic (trunc toward
//            zero, clamp, weights from the CLAMPED x1/y1, add_n order; __fmul_rn/__fadd_rn forbid FMA
//            contraction => bit-identical to the fp32 CPU oracle).
//   phase 3  split mode: results were collected in shared memory as [pixel][plane][channel]; the block writes
//            them out as 16-byte rows (the r01 profile of the direct 2-byte stores: 31 store sectors per unit
//            for 324 useful bytes).  fp32 mode (rb_corr_lookup) stores directly.
// r01 history: v1 one warp per unit, 391 warp instructions per unit, issue-bound; v2 block-cooperative with LDG
// staging, LSU-wavefront-bound (108 wavefronts per unit); v3 = this.
// ---------------------------------------------------------------------------------------------
struct PyramidView {
  const float* base[RB_NUM_LEVELS];
  int hl[RB_NUM_LEVELS], wl[RB_NUM_LEVELS];
  int tma_ok[RB_NUM_LEVELS];  // level rows are 16-byte aligned (W % 4 == 0, aligned base): TMA-stageable
};
struct PyramidMaps {
  CUtensorMap m[RB_NUM_LEVELS];  // (W_l, H_l, B*N) fp32, box (16, 2r+3, 1), 64-byte swizzle
};

constexpr int kLookupPB = 16;    // pixels per block: 440 blocks of 576 threads at 440x1024 = ONE wave at 3 blocks/SM
constexpr int kPatchCols = 16;   // staged columns per row (64 bytes)
constexpr int kUnitBytes = 640;  // shared bytes per unit (>= (2r+2)*64); a multiple of 128 so the swizzle phase is known

// float index of element (row, col) inside a unit's staged patch.  CU_TENSOR_MAP_SWIZZLE_64B XORs the 16-byte chunk
// index with bits [7,9) of the shared-memory byte address = (slot_base/128 + row/2) & 3; `phase` = (slot_base/128) & 3.
__device__ __forceinline__ int patch_idx(int row, int col, int phase) {
  return row * kPatchCols + ((((col >> 2) ^ ((row >> 1) + phase)) & 3) << 2) + (col & 3);
}

__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}

template <int R>
struct LookupSmem {
  static constexpr int D = 2 * R + 1, K = D * D, UNITS = kLookupPB * 4;
  static constexpr int OUTP = (4 * K + 7) / 8 * 8;  // staged channels per pixel and plane (324 -> 328, 196 -> 200)
  static constexpr int kPatchOff = 0;
  static constexpr int kXtabOff = UNITS * kUnitBytes;              // float2 [UNITS][D]: (qx, 4*col of x0 | 4*col of x1 << 8)
  static constexpr int kOutOff = kXtabOff + UNITS * D * 8;         // float [PB][OUTP]: results before the hi/lo split
  static_assert(3 * (kOutOff + kLookupPB * OUTP * 4 + UNITS * 8 + 16 + kLookupPB * 8 + 1024) <= 228 * 1024, "three blocks per SM");
  static constexpr int kBaseOff = kOutOff + kLookupPB * OUTP * 4;  // int [UNITS][2]: bx4, by
  static constexpr int kBarOff = kBaseOff + UNITS * 8;
  static constexpr int kBytes = kBarOff + 16 + kLookupPB * 8;  // + float2 [PB]: the block's coordinates
};

template <int R, bool SPLIT>
__global__ void __launch_bounds__(kLookupPB * 4 * (2 * R + 1), 3)
corr_lookup_kernel(const __grid_constant__ PyramidView pv, const __grid_constant__ PyramidMaps maps,
                   const float2* __restrict__ coords, float* __restrict__ out_f32, __half* __restrict__ out_hi,
                   __half* __restrict__ out_lo, int out_stride, int npix) {
  using L = LookupSmem<R>;
  // P = rows staged per unit: the (2r+2)-row footprint.  The row the fp32 rounding of cy + dy can add (r01 staged it for
  // every unit: +9 % DRAM bytes in a kernel that runs at 80 % of the HBM copy peak at batch 8) is handled by the threads
  // that actually need it with four global loads per tap (`far`, below) -- about one window row in a million.
  constexpr int D = L::D, K = L::K, P = D + 1, UNITS = L::UNITS, NT = UNITS * D, OUTP = L::OUTP;
  extern __shared__ __align__(1024) uint8_t lk_smem[];  // no static shared memory in this kernel: the slots start at 0
  float* patch = reinterpret_cast<float*>(lk_smem + L::kPatchOff);
  float2* xtab = reinterpret_cast<float2*>(lk_smem + L::kXtabOff);
  float* ostage = reinterpret_cast<float*>(lk_smem + L::kOutOff);
  int* ubase = reinterpret_cast<int*>(lk_smem + L::kBaseOff);
  uint64_t* bar = reinterpret_cast<uint64_t*>(lk_smem + L::kBarOff);
  float2* cnew = reinterpret_cast<float2*>(lk_smem + L::kBarOff + 16);  // [PB] coordinates of the block's pixels
  const int tid = threadIdx.x;
  const int pix0 = blockIdx.x * kLookupPB;

  if (tid == 0 && (tc::smem_u32(lk_smem) & 1023u)) __trap();  // the swizzle phase assumes 1024-byte aligned slot 0
  int n_tma = 0;
#pragma unroll
  for (int l = 0; l < 4; ++l) n_tma += pv.tma_ok[l] ? kLookupPB : 0;
  if (tid == 0) {
    tc::mbar_init(bar, 1);
    tc::fence_barrier_init();
    tc::fence_proxy_async();
    if (n_tma) tc::mbar_arrive_expect_tx(bar, (uint32_t)(n_tma * P * kPatchCols * 4));
  }
  if (SPLIT) {  // channel padding of the staged output rows (never produced by a tap)
    for (int e = tid; e < kLookupPB * (OUTP - 4 * K); e += NT) {
      const int row = e / (OUTP - 4 * K), c = 4 * K + e % (OUTP - 4 * K);
      ostage[row * OUTP + c] = 0.f;
    }
  }
  __syncthreads();
  // PDL: dependents may be scheduled from here on (their own griddepcontrol.wait still waits for this grid to finish);
  // nothing above touched global memory, everything below comes after the predecessor kernel.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (tid < kLookupPB) cnew[tid] = __ldg(coords + min(pix0 + tid, npix - 1));  // the block's coordinates, read once
  __syncthreads();
  // ---- phase 0: per-unit origin, TMA issue --------------------------------------------------------------
  // The 64 units are spread over the first lanes of ALL warps: every lane issues its own TMA with its own operands,
  // which ptxas serialises per warp (one elect / R2UR round per distinct lane) -- 4-5 rounds per warp instead of 32 in 2.
  constexpr int kWarps = NT / 32, kUnitsPerWarp = (UNITS + kWarps - 1) / kWarps;
  if ((tid & 31) < kUnitsPerWarp && (tid >> 5) * kUnitsPerWarp + (tid & 31) < UNITS) {
    const int u = (tid >> 5) * kUnitsPerWarp + (tid & 31), pl = u >> 2, lvl = u & 3;
    const int pix = min(pix0 + pl, npix - 1);
    const float2 c = cnew[pl];
    const float inv = 1.0f / (float)(1 << lvl);  // centroid / 2**i (model_utils.py:239), exact
    const int H = pv.hl[lvl], W = pv.wl[lvl];
    const float xf0 = __fadd_rn(c.x * inv, (float)(-R)), yf0 = __fadd_rn(c.y * inv, (float)(-R));
    const int bx4 = min(max((int)xf0, 0), W - 1) & ~3;
    const int by = min(max((int)yf0, 0), H - 1);
    ubase[2 * u] = bx4;
    ubase[2 * u + 1] = by;
    if (pv.tma_ok[lvl]) tc::tma_load_3d(&maps.m[lvl], bar, lk_smem + u * kUnitBytes, bx4, by, pix);
  }
  __syncthreads();
  // ---- fallback staging for levels TMA cannot address (W % 4 != 0) -------------------------------------------
  if (n_tma < UNITS) {
    for (int e = tid; e < UNITS * P * 4; e += NT) {  // one 4-column chunk per thread and round
      const int u = e / (P * 4), rem = e - u * (P * 4), py = rem >> 2, ch = rem & 3;
      const int lvl = u & 3;
      if (pv.tma_ok[lvl]) continue;
      const int pix = min(pix0 + (u >> 2), npix - 1);
      const int H = pv.hl[lvl], W = pv.wl[lvl];
      const int yy = min(ubase[2 * u + 1] + py, H - 1), col = ubase[2 * u] + ch * 4;
      const float* row = pv.base[lvl] + ((size_t)pix * H + yy) * W;
      float4 v;
      v.x = __ldg(row + min(col + 0, W - 1)); v.y = __ldg(row + min(col + 1, W - 1));
      v.z = __ldg(row + min(col + 2, W - 1)); v.w = __ldg(row + min(col + 3, W - 1));
      *reinterpret_cast<float4*>(&patch[u * (kUnitBytes / 4) + patch_idx(py, ch * 4, (u * (kUnitBytes / 128)) & 3)]) = v;
    }
  }
  // ---- phase 1: separable index math ---------------------------------------------------------------------------
  const int u = tid / D, j = tid - u * D;
  const int pl = u >> 2, lvl = u & 3;
  const int pix = pix0 + pl;
  const int H = pv.hl[lvl], W = pv.wl[lvl];
  const float2 c = cnew[pl];
  const float inv = 1.0f / (float)(1 << lvl);
  const float cx = c.x * inv, cy = c.y * inv;
  {
    // x side of window column i = j (i walks x: model_utils.py:235-237)
    const float x = __fadd_rn(cx, (float)(j - R));
    int x0 = (int)x;  // tf.cast truncates toward zero (utils.py:54-57)
    int x1 = x0 + 1;
    x0 = min(max(x0, 0), W - 1);
    x1 = min(max(x1, 0), W - 1);
    const float qx = __fsub_rn((float)x1, x);  // utils.py:84 (clamped x1)
    const int bx4 = ubase[2 * u];
    const int ax0 = min(max(x0 - bx4, 0), kPatchCols - 1), ax1 = min(max(x1 - bx4, 0), kPatchCols - 1);
    xtab[u * D + j] = make_float2(qx, __int_as_float((ax0 * 4) | (ax1 * 4 << 8)));
  }
  const float y = __fadd_rn(cy, (float)(j - R));
  int y0 = (int)y;
  int y1 = y0 + 1;
  y0 = min(max(y0, 0), H - 1);
  y1 = min(max(y1, 0), H - 1);
  const float qy = __fsub_rn((float)y1, y), pyw = __fsub_rn(1.0f, qy);  // utils.py:85
  const int by = ubase[2 * u + 1];
  const bool far = (y1 - by) > P - 1 || (y0 - by) > P - 1;  // rounding slack row outside the staged box
  const int r0 = min(max(y0 - by, 0), P - 1), r1 = min(max(y1 - by, 0), P - 1);
  // Texel address = (swizzled row address) XOR (4 * column): rows are 64 bytes and CU_TENSOR_MAP_SWIZZLE_64B XORs the 16-byte
  // chunk index with ((slot_base / 128 + row / 2) & 3), i.e. only bits 4-5 of the offset inside the row -- so the row part
  // (64-byte aligned address + chunk phase << 4) and the column part (4 * col < 64) combine with ONE xor per texel.
  // (r01 version: ~16 integer instructions of swizzle arithmetic per tap, 75 SASS instructions per tap in total; now 21.)
  const int phase = (u * (kUnitBytes / 128)) & 3;
  const uint32_t ubase_a = tc::smem_u32(lk_smem) + u * kUnitBytes;
  const uint32_t r0a = ubase_a + r0 * 64 + ((((r0 >> 1) + phase) & 3) << 4);
  const uint32_t r1a = ubase_a + r1 * 64 + ((((r1 >> 1) + phase) & 3) << 4);
  __syncthreads();                     // xtab + fallback patches visible
  if (n_tma) tc::mbar_wait(bar, 0);    // TMA patches landed
  // ---- phase 2: taps of window row j ------------------------------------------------------------------------------
  const bool live = pix < npix;
#pragma unroll
  for (int i = 0; i < D; ++i) {
    const float2 xt = xtab[u * D + i];
    const uint32_t pk = (uint32_t)__float_as_int(xt.y), c0 = pk & 0xffu, c1 = pk >> 8;
    const float pxw = __fsub_rn(1.0f, xt.x);
    const float wa = __fmul_rn(xt.x, qy), wb = __fmul_rn(xt.x, pyw);  // utils.py:86-89
    const float wc = __fmul_rn(pxw, qy), wd = __fmul_rn(pxw, pyw);
    float Ia, Ib, Ic, Id;
    if (!far) {
      Ia = lds_f32(r0a ^ c0); Ib = lds_f32(r1a ^ c0); Ic = lds_f32(r0a ^ c1); Id = lds_f32(r1a ^ c1);
    } else {
      const float* img = pv.base[lvl] + (size_t)min(pix, npix - 1) * H * W;
      const int bx4 = ubase[2 * u], xa = bx4 + (int)(c0 >> 2), xb = bx4 + (int)(c1 >> 2);
      Ia = __ldg(img + (size_t)y0 * W + xa); Ib = __ldg(img + (size_t)y1 * W + xa);
      Ic = __ldg(img + (size_t)y0 * W + xb); Id = __ldg(img + (size_t)y1 * W + xb);
    }
    const float v = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(wa, Ia), __fmul_rn(wb, Ib)), __fmul_rn(wc, Ic)),
                              __fmul_rn(wd, Id));  // tf.add_n order (utils.py:98)
    const int ch = lvl * K + i * D + j;
    if constexpr (SPLIT) {
      ostage[pl * OUTP + ch] = v;
    } else {
      if (live) out_f32[(size_t)pix * out_stride + ch] = v;
    }
  }
  // ---- phase 3: hi/lo split of 8 consecutive channels per thread, 16-byte stores per plane ---------------------------------
  if constexpr (SPLIT) {
    __syncthreads();
    constexpr int V = OUTP / 8;  // 8-channel groups per pixel
    for (int e = tid; e < kLookupPB * V; e += NT) {
      const int p2 = e / V, v8 = e - p2 * V;
      if (pix0 + p2 >= npix) continue;
      const float4 a = *reinterpret_cast<const float4*>(ostage + p2 * OUTP + v8 * 8);
      const float4 b = *reinterpret_cast<const float4*>(ostage + p2 * OUTP + v8 * 8 + 4);
      uint4 h, l;
      split2(a.x, a.y, h.x, l.x); split2(a.z, a.w, h.y, l.y);
      split2(b.x, b.y, h.z, l.z); split2(b.z, b.w, h.w, l.w);
      *reinterpret_cast<uint4*>(out_hi + (size_t)(pix0 + p2) * out_stride + v8 * 8) = h;
      *reinterpret_cast<uint4*>(out_lo + (size_t)(pix0 + p2) * out_stride + v8 * 8) = l;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// A2/A3 lookup, warp-per-pixel form ("v5", round 2): the kernel of the VOLUME-FREE path (OTF = true) and an opt-in
// alternative for the materialised volume (RAFT_B200_LOOKUP_V5=1).  What the r01 profile said about the round-1 kernel: 75 SASS instructions per tap (swizzle /
// index arithmetic), 1.86x more DRAM bytes than the algorithmic count (16-column, (2r+3)-row boxes promoted to 256-byte
// L2 requests).  v5:
//   * one WARP per query pixel, its 4 pyramid levels = 4 units; lane = tap (t = i*D + j, ceil(K/32) rounds), so the
//     results of a unit are 32 consecutive words of the staging row (conflict-free) and a unit's patch is read by
//     lanes whose rows land in 8 distinct bank groups under the 64-byte swizzle (conflict-free up to j = 0 / D-1);
//   * the patch of a unit is ONE TMA box of 16 columns x (2r+2) rows fp32 (64-byte swizzle, L2 promotion off) whose origin
//     is (x0 & ~3, y0), (x0, y0) = clamp(trunc(centroid - r)): one row less than v4.  (A 12-column box at the unaligned x0
//     was the first r02 attempt: the TMA unit raises "illegal instruction" when the innermost box coordinate is not a
//     multiple of 16 bytes -- compute-sanitizer log in profiles/r02_notes.md.)  The (2r+2)^2 footprint plus the
//     fp32-rounding slack column fits; a unit whose rounding slack falls outside the box (trunc(fl(c+d)) ==
//     trunc(c-r)+d+1 in the last row) is detected while its index tables are built and takes a per-tap global-load
//     path (warp-uniform branch, ~never taken);
//   * separable index math once per unit: x table {qx, 1-qx, 4*col of x0, of x1} and y table {qy, 1-qy, swizzled row address
//     of y0, of y1} in shared memory (two 128-bit broadcast loads per tap; texel address = row address XOR 4*col, one
//     LOP3), tap arithmetic exactly as the reference
//     (trunc toward zero, clamp, weights from the CLAMPED x1/y1, add_n order, no FMA contraction) => bit-identical;
//   * every warp is self-contained (own mbarrier, own staging row, __syncwarp only): no block-wide barrier after the
//     prologue; the fp16 hi/lo split happens in the output pass on 8 consecutive channels per lane (128-bit stores).
// ---------------------------------------------------------------------------------------------
template <int R, bool OTF = false>
struct LookupV5 {
  // OTF (volume-free, SURVEY 8(f) F2): the patch is COMPUTED (dot products against pooled fmap2), with the slack row included
  static constexpr int D = 2 * R + 1, K = D * D, COLS = 16, ROWS = OTF ? D + 2 : D + 1, PITCH = COLS * 4;
  static constexpr int SLOT = (ROWS * PITCH + 127) / 128 * 128;  // TMA destinations are 128-byte aligned
  static constexpr int PB = 16, WARPS = PB, NT = WARPS * 32, ROUNDS = (K + 31) / 32;
  static constexpr int OUTP = (4 * K + 7) / 8 * 8;  // staged channels per pixel (324 -> 328, 196 -> 200)
  static constexpr int TABN = 2 * D;                // table entries per unit: D x-entries, D y-entries (float4 each)
  static constexpr int kTabOff = PB * 4 * SLOT;
  static constexpr int kStageOff = kTabOff + PB * 4 * TABN * 16;
  static constexpr int kBarOff = kStageOff + PB * OUTP * 4;
  static constexpr int kBytes = kBarOff + 128;
};
// volume-free mode: level l of the pyramid is fmap1 . pool^l(fmap2)^T / sqrt(C) (exact by linearity, gemm_tc.cu); here the
// (2r+3) x 11 entries a unit can touch are evaluated on the fly instead of being read from a materialised volume.
struct OtfView {
  const float* f1;                 // [B,h,w,C]
  const float* f2[RB_NUM_LEVELS];  // pooled fmap2, level l: [B, h>>l, w>>l, C] fp32
  int C, N;                        // channels (<= 256, multiple of 4), pixels per sample (h*w)
};
struct PyramidMapsV5 {
  CUtensorMap m[RB_NUM_LEVELS];  // (W_l, H_l, B*N) fp32, box (16, 2r+2, 1), 64-byte swizzle, no L2 promotion
};
// Byte offset of patch element (row, col) inside a unit whose slot starts `unit_off` bytes after the 1024-byte aligned
// start of shared memory: rows are 64 bytes; CU_TENSOR_MAP_SWIZZLE_64B XORs the 16-byte chunk index with bits [7,9) of the
// shared-memory byte address, i.e. with s(row) = (unit_off / 128 + row / 2) & 3.
__device__ __forceinline__ int v5_row_off(int unit_off, int row) { return row * 64 + ((((unit_off >> 7) + (row >> 1)) & 3) << 4); }

template <int R, bool SPLIT, bool OTF = false>
__global__ void __launch_bounds__(LookupV5<R, OTF>::NT, OTF ? 2 : 3)
corr_lookup_v5_kernel(const __grid_constant__ PyramidView pv, const __grid_constant__ PyramidMapsV5 maps,
                      const float2* __restrict__ coords, float* __restrict__ out_f32, __half* __restrict__ out_hi,
                      __half* __restrict__ out_lo, int out_stride, int npix, const OtfView otf) {
  using L = LookupV5<R, OTF>;
  constexpr int D = L::D, K = L::K;
  extern __shared__ __align__(1024) uint8_t lk5_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int pix = blockIdx.x * L::PB + warp;
  float4* tab = reinterpret_cast<float4*>(lk5_smem + L::kTabOff) + warp * 4 * L::TABN;
  float* stage = reinterpret_cast<float*>(lk5_smem + L::kStageOff) + warp * L::OUTP;
  // ONE mbarrier per block at a block-uniform address (the v4 pattern).  A per-warp barrier has a warp-dependent address:
  // ptxas then emulates mbarrier.init with STS.64 + SYNCS.CCTL.IVALL instead of SYNCS.EXCH, and the first r02 build of this
  // kernel (per-warp barriers) died with "illegal instruction" on the B200 -- not worth the ~1 us of decoupling.
  uint64_t* bar = reinterpret_cast<uint64_t*>(lk5_smem + L::kBarOff);
  uint8_t* patch = lk5_smem + warp * 4 * L::SLOT;
  const uint32_t patch0_u32 = tc::smem_u32(lk5_smem);  // 1024-byte aligned (checked below): slot offsets decide the swizzle
  if (threadIdx.x == 0 && (patch0_u32 & 1023u)) __trap();
  const bool live = pix < npix;

  int n_tma = 0;
#pragma unroll
  for (int l = 0; l < 4; ++l) n_tma += (!OTF && pv.tma_ok[l]) ? 1 : 0;
  if (threadIdx.x == 0) {
    tc::mbar_init(bar, 1);
    tc::fence_barrier_init();
    tc::fence_proxy_async();
    const int live_px = min(L::PB, npix - (int)blockIdx.x * L::PB);  // >= 1: the grid covers npix
    if (n_tma) tc::mbar_arrive_expect_tx(bar, (uint32_t)(live_px * n_tma * L::ROWS * L::PITCH));
  }
  if (lane < L::OUTP - 4 * K) stage[4 * K + lane] = 0.f;  // channel padding of the staged row
  // taps of this lane: t = lane + 32*round = i*D + j   (i walks x, j walks y: model_utils.py:235-237)
  int ti[L::ROUNDS], tj[L::ROUNDS];
#pragma unroll
  for (int rd = 0; rd < L::ROUNDS; ++rd) {
    const int t = lane + 32 * rd;
    ti[rd] = t / D;
    tj[rd] = t - ti[rd] * D;
  }
  __syncthreads();  // barrier initialised before any warp can issue a TMA that signals it (the only block-wide barrier)
  // PDL: dependents may be scheduled from here on (their own griddepcontrol.wait still waits for this grid to finish);
  // nothing above touched global memory, everything below comes after the predecessor kernel.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (!live) return;  // warp-uniform; no block-wide barrier below

  const float2 c = __ldg(coords + pix);
  // ---- unit origins (lanes 0..3 hold the values of unit k = lane) and TMA issue ----------------------------------------
  int bx, by;
  {
    const int k = lane & 3;
    const float inv = 1.0f / (float)(1 << k);  // centroid / 2**i (model_utils.py:239), exact
    const int H = pv.hl[k], W = pv.wl[k];
    bx = min(max((int)__fadd_rn(c.x * inv, (float)(-R)), 0), W - 1);
    by = min(max((int)__fadd_rn(c.y * inv, (float)(-R)), 0), H - 1);
    if (!OTF) bx &= ~3;  // TMA: the innermost box coordinate must be a multiple of 16 bytes
    if (!OTF && lane < 4 && pv.tma_ok[k]) tc::tma_load_3d(&maps.m[k], bar, patch + k * L::SLOT, bx, by, pix);
  }
  // ---- index tables: lane -> (unit k = lane >> 3, entry e = lane & 7); entry 8 (r = 4) by the lanes with e = 0 / 1 ------
  unsigned bad = 0;
  {
    const int k = lane >> 3, e = lane & 7;
    const int bxk = __shfl_sync(0xffffffffu, bx, k), byk = __shfl_sync(0xffffffffu, by, k);
    const float inv = 1.0f / (float)(1 << k);
    const float cx = c.x * inv, cy = c.y * inv;
    const int H = pv.hl[k], W = pv.wl[k];
    auto x_entry = [&](int i) {
      const float x = __fadd_rn(cx, (float)(i - R));
      int x0 = (int)x;  // tf.cast truncates toward zero (utils.py:54-57)
      int x1 = x0 + 1;
      x0 = min(max(x0, 0), W - 1);
      x1 = min(max(x1, 0), W - 1);
      const float qx = __fsub_rn((float)x1, x);  // utils.py:84 (clamped x1)
      const int a0 = x0 - bxk, a1 = x1 - bxk;
      if ((unsigned)a0 >= (unsigned)L::COLS || (unsigned)a1 >= (unsigned)L::COLS) bad = 1;
      tab[k * L::TABN + i] = make_float4(qx, __fsub_rn(1.0f, qx), __int_as_float(a0 * 4), __int_as_float(a1 * 4));
    };
    auto y_entry = [&](int j) {
      const float y = __fadd_rn(cy, (float)(j - R));
      int y0 = (int)y;
      int y1 = y0 + 1;
      y0 = min(max(y0, 0), H - 1);
      y1 = min(max(y1, 0), H - 1);
      const float qy = __fsub_rn((float)y1, y);  // utils.py:85
      const int r0 = y0 - byk, r1 = y1 - byk;
      if ((unsigned)r0 >= (unsigned)L::ROWS || (unsigned)r1 >= (unsigned)L::ROWS) bad = 1;
      const int uoff = (warp * 4 + k) * L::SLOT;  // slot offset from the 1024-byte aligned start of shared memory
      tab[k * L::TABN + D + j] = make_float4(qy, __fsub_rn(1.0f, qy), __int_as_float((int)patch0_u32 + uoff + v5_row_off(uoff, r0)),
                                             __int_as_float((int)patch0_u32 + uoff + v5_row_off(uoff, r1)));
    };
    if (e < D) { x_entry(e); y_entry(e); }
    if (D > 8) {
      if (e == 0) x_entry(8);
      if (e == 1) y_entry(8);
    }
  }
  const unsigned badmask = __ballot_sync(0xffffffffu, bad != 0);  // bits 8k..8k+7 belong to unit k
  // ---- volume-free mode: evaluate the patch entries ----------------------------------------------------------------------
  // The warp reads each target feature row COALESCED (lane = 4 channels per 128-channel half; fmap1[pix] stays in 8
  // registers), 8 entries at a time, and reduces the 8 x 32 partial sums with a recursive-halving exchange (9 shuffles per 8
  // entries).  First version (lane = entry, each lane streaming its own 1 KB row): 32 L1 lines per load instruction, 2x
  // sector waste, 1.3 ms per lookup at 55x128 -- L2-bound; neighbouring pixels share most rows, which this form lets L1 see.
  if constexpr (OTF) {
    const int C = otf.C;
    const bool two = C > 128;  // C is 128 or 256 (launch_lookup_otf)
    const float4 fa = __ldg(reinterpret_cast<const float4*>(otf.f1 + (size_t)pix * C + 4 * lane));
    const float4 fb = two ? __ldg(reinterpret_cast<const float4*>(otf.f1 + (size_t)pix * C + 128 + 4 * lane)) : make_float4(0.f, 0.f, 0.f, 0.f);
    const int b = pix / otf.N;
    const float sq = sqrtf((float)C);
    constexpr int NE = L::ROWS * 11;  // columns 0..10 (= D+1 + rounding slack at r = 4) can be indexed
#pragma unroll 1
    for (int k = 0; k < 4; ++k) {
      const int bxk = __shfl_sync(0xffffffffu, bx, k), byk = __shfl_sync(0xffffffffu, by, k);
      const int H = pv.hl[k], W = pv.wl[k];
      const float* f2b = otf.f2[k] + (size_t)b * H * W * C + 4 * lane;
#pragma unroll 1
      for (int e0 = 0; e0 < NE; e0 += 8) {
        float p[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int e = min(e0 + u, NE - 1);
          const int row = e / 11, col = e - row * 11;
          const float* src = f2b + ((size_t)min(byk + row, H - 1) * W + min(bxk + col, W - 1)) * C;
          const float4 v = __ldg(reinterpret_cast<const float4*>(src));
          float acc = fmaf(fa.w, v.w, fmaf(fa.z, v.z, fmaf(fa.y, v.y, fa.x * v.x)));
          if (two) {
            const float4 v2 = __ldg(reinterpret_cast<const float4*>(src + 128));
            acc = fmaf(fb.w, v2.w, fmaf(fb.z, v2.z, fmaf(fb.y, v2.y, fmaf(fb.x, v2.x, acc))));
          }
          p[u] = acc;
        }
        {  // 8 -> 4 -> 2 -> 1 values per lane (partners at xor 16, 8, 4), then the last two steps of a plain butterfly
          const bool up = (lane & 16) != 0;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float keep = up ? p[i + 4] : p[i], send = up ? p[i] : p[i + 4];
            p[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
          }
        }
        {
          const bool up = (lane & 8) != 0;
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const float keep = up ? p[i + 2] : p[i], send = up ? p[i] : p[i + 2];
            p[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
          }
        }
        {
          const bool up = (lane & 4) != 0;
          const float keep = up ? p[1] : p[0], send = up ? p[0] : p[1];
          p[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
        p[0] += __shfl_xor_sync(0xffffffffu, p[0], 2);
        p[0] += __shfl_xor_sync(0xffffffffu, p[0], 1);
        const int e = e0 + ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
        if ((lane & 3) == 0 && e < NE) {
          const int row = e / 11, col = e - row * 11;
          const int uoff = (warp * 4 + k) * L::SLOT;
          *reinterpret_cast<float*>(lk5_smem + uoff + (v5_row_off(uoff, row) ^ (col * 4))) = __fdiv_rn(p[0], sq);  // divide AFTER the matmul (:213)
        }
      }
    }
  }
  // ---- levels TMA cannot address (W % 4 != 0): plain loads into the same layout ------------------------------------------
  if (!OTF && n_tma < 4) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (pv.tma_ok[k]) continue;
      const int bxk = __shfl_sync(0xffffffffu, bx, k), byk = __shfl_sync(0xffffffffu, by, k);
      const int H = pv.hl[k], W = pv.wl[k];
      const int uoff = (warp * 4 + k) * L::SLOT;
      for (int e = lane; e < L::ROWS * 4; e += 32) {
        const int row = e >> 2, ch = e & 3;
        const float* src = pv.base[k] + ((size_t)pix * H + min(byk + row, H - 1)) * W;
        const int col = bxk + ch * 4;
        float4 v;
        v.x = __ldg(src + min(col + 0, W - 1)); v.y = __ldg(src + min(col + 1, W - 1));
        v.z = __ldg(src + min(col + 2, W - 1)); v.w = __ldg(src + min(col + 3, W - 1));
        *reinterpret_cast<float4*>(lk5_smem + uoff + (v5_row_off(uoff, row) ^ (ch * 16))) = v;
      }
    }
  }
  __syncwarp();  // tables and fallback patches visible to the warp
  if (n_tma) tc::mbar_wait(bar, 0);  // all patches of the block have landed
  // ---- taps -----------------------------------------------------------------------------------------------------------------
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int bxk = __shfl_sync(0xffffffffu, bx, k), byk = __shfl_sync(0xffffffffu, by, k);  // converged here (slow path only)
    const float4* xt = tab + k * L::TABN;
    const float4* yt = xt + D;
    const bool slow = ((badmask >> (8 * k)) & 0xffu) != 0;  // warp-uniform
#pragma unroll
    for (int rd = 0; rd < L::ROUNDS; ++rd) {
      const int t = lane + 32 * rd;
      if (t < K) {
        const float4 X = xt[ti[rd]], Y = yt[tj[rd]];
        const float wa = __fmul_rn(X.x, Y.x), wb = __fmul_rn(X.x, Y.y);  // utils.py:86-89
        const float wc = __fmul_rn(X.y, Y.x), wd = __fmul_rn(X.y, Y.y);
        const int a0 = __float_as_int(X.z), a1 = __float_as_int(X.w), r0 = __float_as_int(Y.z), r1 = __float_as_int(Y.w);
        float Ia, Ib, Ic, Id;
        if (OTF || !slow) {  // r0 / r1: swizzled row addresses (64-byte aligned + chunk phase), a0 / a1: 4 * column
          Ia = lds_f32(r0 ^ a0); Ib = lds_f32(r1 ^ a0);
          Ic = lds_f32(r0 ^ a1); Id = lds_f32(r1 ^ a1);
        } else {  // rounding slack outside the box: read the four texels from the volume itself
          const int H = pv.hl[k], W = pv.wl[k];
          const float* img = pv.base[k] + (size_t)pix * H * W;
          const int ubase = (int)patch0_u32 + (warp * 4 + k) * L::SLOT;
          const int x0 = bxk + (a0 >> 2), x1 = bxk + (a1 >> 2), y0 = byk + ((r0 - ubase) >> 6), y1 = byk + ((r1 - ubase) >> 6);
          Ia = __ldg(img + (size_t)y0 * W + x0); Ib = __ldg(img + (size_t)y1 * W + x0);
          Ic = __ldg(img + (size_t)y0 * W + x1); Id = __ldg(img + (size_t)y1 * W + x1);
        }
        stage[k * K + t] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(wa, Ia), __fmul_rn(wb, Ib)), __fmul_rn(wc, Ic)),
                                     __fmul_rn(wd, Id));  // tf.add_n order (utils.py:98)
      }
    }
  }
  __syncwarp();
  // ---- output pass: this warp's pixel, 8 consecutive channels per lane --------------------------------------------------------
  if constexpr (SPLIT) {
    for (int g = lane; g < L::OUTP / 8; g += 32) {
      const float4 v0 = *reinterpret_cast<const float4*>(stage + g * 8);
      const float4 v1 = *reinterpret_cast<const float4*>(stage + g * 8 + 4);
      uint4 h, l;
      split2(v0.x, v0.y, h.x, l.x); split2(v0.z, v0.w, h.y, l.y);
      split2(v1.x, v1.y, h.z, l.z); split2(v1.z, v1.w, h.w, l.w);
      *reinterpret_cast<uint4*>(out_hi + (size_t)pix * out_stride + g * 8) = h;
      *reinterpret_cast<uint4*>(out_lo + (size_t)pix * out_stride + g * 8) = l;
    }
  } else {
    for (int g = lane; g < K; g += 32)  // 4*K floats = K float4 (out_stride = 4*K, 16-byte aligned rows)
      *reinterpret_cast<float4*>(out_f32 + (size_t)pix * out_stride + g * 4) = *reinterpret_cast<const float4*>(stage + g * 4);
  }
}

// General form of bilinear_sampler / tf_grid_sample (utils.py:39-103) for single-channel images:
// img [n,H,W,1], coords [n,S,2] -> out [n,S].  One thread per sample; same arithmetic as above.
__global__ void bilinear_sample_kernel(const float* __restrict__ img, const float2* __restrict__ coords,
                                       float* __restrict__ out, int n, int H, int W, int S) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)n * S) return;
  const float* im = img + (i / S) * (size_t)H * W;
  const float2 c = coords[i];
  int x0 = (int)c.x, y0 = (int)c.y;
  int x1 = x0 + 1, y1 = y0 + 1;
  x0 = min(max(x0, 0), W - 1); x1 = min(max(x1, 0), W - 1);
  y0 = min(max(y0, 0), H - 1); y1 = min(max(y1, 0), H - 1);
  const float qx = __fsub_rn((float)x1, c.x), qy = __fsub_rn((float)y1, c.y);
  const float pxw = __fsub_rn(1.0f, qx), pyw = __fsub_rn(1.0f, qy);
  const float Ia = im[(size_t)y0 * W + x0], Ib = im[(size_t)y1 * W + x0];
  const float Ic = im[(size_t)y0 * W + x1], Id = im[(size_t)y1 * W + x1];
  out[i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(__fmul_rn(qx, qy), Ia), __fmul_rn(__fmul_rn(qx, pyw), Ib)),
                               __fmul_rn(__fmul_rn(pxw, qy), Ic)),
                     __fmul_rn(__fmul_rn(pxw, pyw), Id));
}

int pyramid_view(const float* pyramid, int B, int h, int w, PyramidView* pv) {
  size_t off = 0;
  size_t rows = (size_t)B * h * w;
  for (int l = 0; l < RB_NUM_LEVELS; ++l) {
    int hl = level_dim(h, l), wl = level_dim(w, l);
    if (hl < 1 || wl < 1) {
      set_error("pyramid level %d is empty for a %dx%d grid", l, h, w);
      return RB_ERR_BAD_SHAPE;
    }
    pv->base[l] = pyramid + off;
    pv->hl[l] = hl;
    pv->wl[l] = wl;
    pv->tma_ok[l] = (wl % 4 == 0) && (reinterpret_cast<uintptr_t>(pyramid + off) % 16 == 0);
    off += rows * hl * wl;
  }
  return RB_OK;
}

template <int R>
static size_t lookup_smem_bytes() {
  return (size_t)LookupSmem<R>::kBytes;
}

template <int R, bool SPLIT>
static int launch_lookup_cfg(const PyramidView& pv, const PyramidMaps& maps, const float2* c2, float* out_f32, __half* out_hi,
                             __half* out_lo, int out_stride, int npix, cudaStream_t s) {
  static PerDeviceOnce attr_set;
  const size_t smem = lookup_smem_bytes<R>();
  int dev = 0, rc_dev;
  if ((rc_dev = current_device(&dev))) return rc_dev;
  if (!attr_set.test(dev)) {
    RB_CHECK_CUDA(cudaFuncSetAttribute(corr_lookup_kernel<R, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set.set(dev);
  }
  dim3 grid((npix + kLookupPB - 1) / kLookupPB), block(kLookupPB * 4 * (2 * R + 1));
  // Programmatic dependent launch (as the convs, conv_tc.cu): inside the iteration loop the lookup follows the flow-head
  // conv and precedes convc1; its blocks are scheduled while the predecessor drains and wait in griddepcontrol.wait
  // before they read the coordinates.
  static const int pdl = getenv("RAFT_B200_NO_PDL") ? 0 : 1;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl;
  RB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, corr_lookup_kernel<R, SPLIT>, pv, maps, c2, out_f32, out_hi, out_lo, out_stride, npix));
  RB_CHECK_LAUNCH("corr_lookup_kernel");
  return RB_OK;
}

template <int R, bool SPLIT, bool OTF = false>
static int launch_lookup_v5(const PyramidView& pv, const PyramidMapsV5& maps, const float2* c2, float* out_f32, __half* out_hi,
                            __half* out_lo, int out_stride, int npix, cudaStream_t s, const OtfView& otf = OtfView{}) {
  using L = LookupV5<R, OTF>;
  static PerDeviceOnce attr_set;
  int dev = 0, rc_dev;
  if ((rc_dev = current_device(&dev))) return rc_dev;
  if (!attr_set.test(dev)) {
    RB_CHECK_CUDA(cudaFuncSetAttribute(corr_lookup_v5_kernel<R, SPLIT, OTF>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kBytes));
    attr_set.set(dev);
  }
  static const int pdl = getenv("RAFT_B200_NO_PDL") ? 0 : 1;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((npix + L::PB - 1) / L::PB);
  cfg.blockDim = dim3(L::NT);
  cfg.dynamicSmemBytes = L::kBytes;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl;
  RB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, corr_lookup_v5_kernel<R, SPLIT, OTF>, pv, maps, c2, out_f32, out_hi, out_lo, out_stride, npix, otf));
  RB_CHECK_LAUNCH("corr_lookup_v5_kernel");
  return RB_OK;
}

int launch_lookup(const float* pyramid, const float* coords, float* out_f32, __half* out_hi,
                  __half* out_lo, int out_stride, int B, int h, int w, int radius, cudaStream_t s) {
  PyramidView pv;
  int rc = pyramid_view(pyramid, B, h, w, &pv);
  if (rc) return rc;
  RB_REQUIRE(radius == 3 || radius == 4, RB_ERR_UNSUPPORTED, "radius %d unsupported (3 = raft-small, 4 = raft-things)", radius);
  RB_REQUIRE(out_hi == nullptr || out_stride % 8 == 0, RB_ERR_BAD_SHAPE, "lookup: split output stride %d not a multiple of 8",
             out_stride);
  const int npix = B * h * w;
  const float2* c2 = reinterpret_cast<const float2*>(coords);
  const bool split = out_hi != nullptr;
  // Default: corr_lookup_kernel (block = 16 px x 4 levels, thread = window row).  RAFT_B200_LOOKUP_V5=1 selects the
  // warp-per-pixel kernel (lane = tap) that the volume-free path is built on: same DRAM traffic, 29 % shared-memory bank
  // conflicts (nine window rows of one column can never sit in nine distinct bank groups) -- 14 % slower at batch 8
  // (profiles/r02_notes.md), kept selectable because it shares every line with the volume-free instantiation.
  static const bool v5 = getenv("RAFT_B200_LOOKUP_V5") != nullptr;
  const bool f32_rows_ok = split || (out_stride % 4 == 0 && reinterpret_cast<uintptr_t>(out_f32) % 16 == 0);
  if (v5 && f32_rows_ok) {
    PyramidMapsV5 maps;
    memset(&maps, 0, sizeof(maps));
    for (int l = 0; l < RB_NUM_LEVELS; ++l) {
      if (!pv.tma_ok[l]) continue;
      uint64_t dims[3] = {(uint64_t)pv.wl[l], (uint64_t)pv.hl[l], (uint64_t)npix};
      uint64_t str[2] = {(uint64_t)pv.wl[l] * 4, (uint64_t)pv.wl[l] * pv.hl[l] * 4};
      uint32_t box[3] = {16u, (uint32_t)(2 * radius + 2), 1};
      if (cached_tmap(&maps.m[l], pv.base[l], 3, dims, str, box, tc::TMAP_F32_SW64_GATHER) != RB_OK) pv.tma_ok[l] = 0;  // plain loads
    }
    if (radius == 4)
      return split ? launch_lookup_v5<4, true>(pv, maps, c2, nullptr, out_hi, out_lo, out_stride, npix, s)
                   : launch_lookup_v5<4, false>(pv, maps, c2, out_f32, nullptr, nullptr, out_stride, npix, s);
    return split ? launch_lookup_v5<3, true>(pv, maps, c2, nullptr, out_hi, out_lo, out_stride, npix, s)
                 : launch_lookup_v5<3, false>(pv, maps, c2, out_f32, nullptr, nullptr, out_stride, npix, s);
  }
  PyramidMaps maps;
  memset(&maps, 0, sizeof(maps));
  for (int l = 0; l < RB_NUM_LEVELS; ++l) {
    if (!pv.tma_ok[l]) continue;
    uint64_t dims[3] = {(uint64_t)pv.wl[l], (uint64_t)pv.hl[l], (uint64_t)npix};
    uint64_t str[2] = {(uint64_t)pv.wl[l] * 4, (uint64_t)pv.wl[l] * pv.hl[l] * 4};
    uint32_t box[3] = {(uint32_t)kPatchCols, (uint32_t)(2 * radius + 2), 1};
    if (cached_tmap(&maps.m[l], pv.base[l], 3, dims, str, box, tc::TMAP_F32_SW64) != RB_OK) pv.tma_ok[l] = 0;  // plain loads instead
  }
  if (radius == 4)
    return split ? launch_lookup_cfg<4, true>(pv, maps, c2, nullptr, out_hi, out_lo, out_stride, npix, s)
                 : launch_lookup_cfg<4, false>(pv, maps, c2, out_f32, nullptr, nullptr, out_stride, npix, s);
  return split ? launch_lookup_cfg<3, true>(pv, maps, c2, nullptr, out_hi, out_lo, out_stride, npix, s)
               : launch_lookup_cfg<3, false>(pv, maps, c2, out_f32, nullptr, nullptr, out_stride, npix, s);
}

// ---- F2: volume-free correlation ---------------------------------------------------------------------------------------------
// workspace = pooled fmap2 levels 1..3 (fp32); level 0 is the caller's fmap2 itself
static size_t otf_level_offset(int B, int h, int w, int C, int level) {  // floats; level 1..4 (4 = total)
  size_t off = 0;
  for (int l = 1; l < level; ++l) off += (size_t)B * level_dim(h, l) * level_dim(w, l) * C;
  return off;
}
__global__ void otf_pool_kernel(const float* __restrict__ src, float* __restrict__ dst, int B, int hs, int ws, int hd, int wd, int C) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // 2x2 VALID average pool of an NHWC map (model_utils.py:217-219 by linearity)
  if (i >= (size_t)B * hd * wd * C) return;
  int c = i % C;
  size_t t = i / C;
  int x = t % wd; t /= wd;
  int y = t % hd;
  int b = t / hd;
  const float* p = src + (((size_t)b * hs + 2 * y) * ws + 2 * x) * C + c;
  dst[i] = (p[0] + p[C] + p[(size_t)ws * C] + p[(size_t)ws * C + C]) * 0.25f;
}
int launch_lookup_otf(const float* fmap1, const float* fmap2, const float* pooled, const float* coords, float* out_f32,
                      __half* out_hi, __half* out_lo, int out_stride, int B, int h, int w, int C, int radius, cudaStream_t s) {
  RB_REQUIRE(radius == 3 || radius == 4, RB_ERR_UNSUPPORTED, "radius %d unsupported", radius);
  RB_REQUIRE(C == 128 || C == 256, RB_ERR_BAD_SHAPE, "volume-free lookup: C=%d (128 = raft-small, 256 = raft-things)", C);
  RB_REQUIRE((h >> 3) >= 1 && (w >> 3) >= 1, RB_ERR_BAD_SHAPE, "volume-free lookup: grid %dx%d too small for 4 levels", h, w);
  RB_REQUIRE(out_hi == nullptr || out_stride % 8 == 0, RB_ERR_BAD_SHAPE, "lookup: split output stride %d", out_stride);
  PyramidView pv;
  memset(&pv, 0, sizeof(pv));
  OtfView otf;
  otf.f1 = fmap1; otf.C = C; otf.N = h * w;
  for (int l = 0; l < RB_NUM_LEVELS; ++l) {
    pv.hl[l] = level_dim(h, l); pv.wl[l] = level_dim(w, l);
    otf.f2[l] = l == 0 ? fmap2 : pooled + otf_level_offset(B, h, w, C, l);
  }
  PyramidMapsV5 maps;
  memset(&maps, 0, sizeof(maps));
  const float2* c2 = reinterpret_cast<const float2*>(coords);
  const int npix = B * h * w;
  const bool split = out_hi != nullptr;
  if (radius == 4)
    return split ? launch_lookup_v5<4, true, true>(pv, maps, c2, nullptr, out_hi, out_lo, out_stride, npix, s, otf)
                 : launch_lookup_v5<4, false, true>(pv, maps, c2, out_f32, nullptr, nullptr, out_stride, npix, s, otf);
  return split ? launch_lookup_v5<3, true, true>(pv, maps, c2, nullptr, out_hi, out_lo, out_stride, npix, s, otf)
               : launch_lookup_v5<3, false, true>(pv, maps, c2, out_f32, nullptr, nullptr, out_stride, npix, s, otf);
}

int corr_build_tc(const float* fmap1, const float* fmap2, float* pyramid, int B, int h, int w, int C,
                  void* ws, size_t ws_bytes, cudaStream_t s);
size_t corr_tc_workspace_bytes(int B, int h, int w, int C);

}  // namespace rb

using namespace rb;

extern "C" int rb_coords_grid(float* coords, int B, int h, int w, void* stream) {
  RB_REQUIRE(coords && B > 0 && h > 0 && w > 0, RB_ERR_BAD_ARG, "rb_coords_grid: bad argument");
  int n = B * h * w;
  coords_grid_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<float2*>(coords), B, h, w);
  RB_CHECK_LAUNCH("coords_grid_kernel");
  return RB_OK;
}

extern "C" int rb_corr_level_offset(int B, int h, int w, int level, size_t* offset_floats, int* hl, int* wl) {
  RB_REQUIRE(B > 0 && h > 0 && w > 0 && level >= 0 && level <= RB_NUM_LEVELS, RB_ERR_BAD_ARG,
             "rb_corr_level_offset: bad argument");
  size_t off = 0, rows = (size_t)B * h * w;
  for (int l = 0; l < level; ++l) off += rows * level_dim(h, l) * level_dim(w, l);
  if (offset_floats) *offset_floats = off;
  if (hl) *hl = level < RB_NUM_LEVELS ? level_dim(h, level) : 0;
  if (wl) *wl = level < RB_NUM_LEVELS ? level_dim(w, level) : 0;
  return RB_OK;
}

extern "C" int rb_corr_pyramid_bytes(int B, int h, int w, size_t* bytes) {
  RB_REQUIRE(bytes, RB_ERR_BAD_ARG, "rb_corr_pyramid_bytes: null output");
  RB_REQUIRE(B > 0 && (h >> 3) >= 1 && (w >> 3) >= 1, RB_ERR_BAD_SHAPE,
             "rb_corr_pyramid_bytes: grid %dx%d too small for 4 levels", h, w);
  size_t off;
  rb_corr_level_offset(B, h, w, RB_NUM_LEVELS, &off, nullptr, nullptr);
  *bytes = off * sizeof(float) + 256;  // tail padding: the lookup stages 16-column row segments with vector loads
  return RB_OK;
}

extern "C" int rb_corr_workspace_bytes(int B, int h, int w, int C, size_t* bytes) {
  RB_REQUIRE(bytes && B > 0 && h > 0 && w > 0 && C > 0, RB_ERR_BAD_ARG, "rb_corr_workspace_bytes: bad argument");
  *bytes = corr_tc_workspace_bytes(B, h, w, C);
  return RB_OK;
}

extern "C" int rb_corr_build(const float* fmap1, const float* fmap2, float* pyramid, int B, int h, int w,
                             int C, void* workspace, size_t workspace_bytes, void* stream) {
  RB_REQUIRE(fmap1 && fmap2 && pyramid, RB_ERR_BAD_ARG, "rb_corr_build: null pointer");
  RB_REQUIRE(B > 0 && (h >> 3) >= 1 && (w >> 3) >= 1, RB_ERR_BAD_SHAPE, "rb_corr_build: grid %dx%d too small", h, w);
  RB_REQUIRE(C > 0 && C % 16 == 0, RB_ERR_BAD_SHAPE, "rb_corr_build: C=%d must be a multiple of 16", C);
  cudaStream_t s = (cudaStream_t)stream;
  if (math_mode() == RB_MATH_TC) return corr_build_tc(fmap1, fmap2, pyramid, B, h, w, C, workspace, workspace_bytes, s);
  const int N = h * w;
  dim3 grid((N + 63) / 64, (N + 63) / 64, B);
  corr_gemm_simt_kernel<<<grid, 256, 0, s>>>(fmap1, fmap2, pyramid, N, C, 0.f);
  RB_CHECK_LAUNCH("corr_gemm_simt_kernel");
  size_t rows = (size_t)B * N;
  for (int l = 0; l + 1 < RB_NUM_LEVELS; ++l) {
    size_t so, dofs;
    int hs, ws, hd, wd;
    rb_corr_level_offset(B, h, w, l, &so, &hs, &ws);
    rb_corr_level_offset(B, h, w, l + 1, &dofs, &hd, &wd);
    size_t total = rows * hd * wd;
    avgpool2_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(pyramid + so, pyramid + dofs, rows, hs, ws, hd, wd);
    RB_CHECK_LAUNCH("avgpool2_kernel");
  }
  return RB_OK;
}

extern "C" int rb_bilinear_sample(const float* img, const float* coords, float* out, int n, int H, int W, int S,
                                  void* stream) {
  RB_REQUIRE(img && coords && out, RB_ERR_BAD_ARG, "rb_bilinear_sample: null pointer");
  RB_REQUIRE(n > 0 && H > 0 && W > 0 && S > 0, RB_ERR_BAD_SHAPE, "rb_bilinear_sample: bad shape");
  size_t total = (size_t)n * S;
  bilinear_sample_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      img, reinterpret_cast<const float2*>(coords), out, n, H, W, S);
  RB_CHECK_LAUNCH("bilinear_sample_kernel");
  return RB_OK;
}

extern "C" int rb_corr_lookup(const float* pyramid, const float* coords, float* out, int B, int h, int w,
                              int radius, void* stream) {
  RB_REQUIRE(pyramid && coords && out, RB_ERR_BAD_ARG, "rb_corr_lookup: null pointer");
  RB_REQUIRE(B > 0 && h > 0 && w > 0, RB_ERR_BAD_SHAPE, "rb_corr_lookup: bad shape");
  int K = (2 * radius + 1) * (2 * radius + 1);
  return launch_lookup(pyramid, coords, out, nullptr, nullptr, 4 * K, B, h, w, radius, (cudaStream_t)stream);
}

/* ---- F2: volume-free correlation (SURVEY 8(f)); same results as rb_corr_build + rb_corr_lookup up to fp32 summation order ---- */
extern "C" int rb_corr_otf_workspace_bytes(int B, int h, int w, int C, size_t* bytes) {
  RB_REQUIRE(bytes && B > 0 && h > 0 && w > 0 && C > 0, RB_ERR_BAD_ARG, "rb_corr_otf_workspace_bytes: bad argument");
  *bytes = otf_level_offset(B, h, w, C, RB_NUM_LEVELS) * sizeof(float) + 256;
  return RB_OK;
}

extern "C" int rb_corr_otf_prepare(const float* fmap2, void* workspace, size_t workspace_bytes, int B, int h, int w, int C,
                                   void* stream) {
  RB_REQUIRE(fmap2 && workspace, RB_ERR_BAD_ARG, "rb_corr_otf_prepare: null pointer");
  RB_REQUIRE(B > 0 && (h >> 3) >= 1 && (w >> 3) >= 1 && C > 0, RB_ERR_BAD_SHAPE, "rb_corr_otf_prepare: bad shape");
  size_t need;
  rb_corr_otf_workspace_bytes(B, h, w, C, &need);
  RB_REQUIRE(workspace_bytes >= need, RB_ERR_WORKSPACE, "rb_corr_otf_prepare: workspace has %zu bytes, need %zu", workspace_bytes, need);
  float* pooled = reinterpret_cast<float*>(workspace);
  const float* prev = fmap2;
  for (int l = 1; l < RB_NUM_LEVELS; ++l) {
    float* dst = pooled + otf_level_offset(B, h, w, C, l);
    const int hd = level_dim(h, l), wd = level_dim(w, l);
    const size_t n = (size_t)B * hd * wd * C;
    otf_pool_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(prev, dst, B, level_dim(h, l - 1), level_dim(w, l - 1),
                                                                                 hd, wd, C);
    RB_CHECK_LAUNCH("otf_pool_kernel");
    prev = dst;
  }
  return RB_OK;
}

extern "C" int rb_corr_otf_lookup(const float* fmap1, const float* fmap2, const void* workspace, const float* coords, float* out,
                                  int B, int h, int w, int C, int radius, void* stream) {
  RB_REQUIRE(fmap1 && fmap2 && workspace && coords && out, RB_ERR_BAD_ARG, "rb_corr_otf_lookup: null pointer");
  RB_REQUIRE(B > 0 && h > 0 && w > 0, RB_ERR_BAD_SHAPE, "rb_corr_otf_lookup: bad shape");
  const int K = (2 * radius + 1) * (2 * radius + 1);
  return launch_lookup_otf(fmap1, fmap2, reinterpret_cast<const float*>(workspace), coords, out, nullptr, nullptr, 4 * K, B, h, w, C,
                           radius, (cudaStream_t)stream);
}
