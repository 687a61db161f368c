// Shared declarations for the raft_b200 kernels: status codes, the fp16 hi/lo "split" operand
// format, the conv launch descriptor and the fused epilogues every conv back end shares.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/raft_b200.h"

namespace rb {

// ---- error plumbing ---------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch();
int math_mode();

// Function attributes (cudaFuncAttributeMaxDynamicSharedMemorySize) and the SM count are PER DEVICE: a process may
// drive several GPUs (RaftEngine(device=...)), so "already set" is tracked per (call site, device ordinal).
struct PerDeviceOnce {
  unsigned long long done[4] = {0, 0, 0, 0};  // bit per device ordinal (<= 256 devices); racing first calls are idempotent
  bool test(int dev) const { return (__atomic_load_n(&done[(dev >> 6) & 3], __ATOMIC_ACQUIRE) >> (dev & 63)) & 1ull; }
  void set(int dev) { __atomic_fetch_or(&done[(dev >> 6) & 3], 1ull << (dev & 63), __ATOMIC_RELEASE); }
};
int current_device(int* dev);   // cudaGetDevice with error plumbing
int device_sm_count(int dev);   // cached cudaDevAttrMultiProcessorCount (148 on B200)

#define RB_CHECK_CUDA(expr)                                                                   \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      rb::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return RB_ERR_CUDA;                                                                     \
    }                                                                                         \
  } while (0)

#define RB_CHECK_LAUNCH(name)                                                     \
  do {                                                                            \
    rb::count_launch();                                                           \
    cudaError_t _e = cudaGetLastError();                                          \
    if (_e != cudaSuccess) {                                                      \
      rb::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));     \
      return RB_ERR_CUDA;                                                         \
    }                                                                             \
  } while (0)

#define RB_REQUIRE(cond, code, ...)   \
  do {                                \
    if (!(cond)) {                    \
      rb::set_error(__VA_ARGS__);     \
      return code;                    \
    }                                 \
  } while (0)

// ---- split operand format ---------------------------------------------------------------------
// An fp32 value a is carried as two fp16 numbers: hi = fp16(a) and lo = fp16((a - hi) * 2^11).
// a ~= hi + lo * 2^-11 to ~22 mantissa bits.  A product a*b is evaluated as
//   hi_a*hi_b + 2^-11 * (hi_a*lo_b + lo_a*hi_b)          (the lo*lo term, 2^-22, is dropped)
// with both sums accumulated in fp32: three fp16 tensor-core MMAs per product, two accumulators.
constexpr float kLoScale = 2048.0f;
constexpr float kLoInv = 1.0f / 2048.0f;

// Range: fp16 planes hold |a| <= 65504.  Larger magnitudes SATURATE (finite, wrong) instead of turning into inf -> NaN
// through the tensor-core path; the host side refuses weights outside the range (raft_b200/weights.py) and the engine
// checks the fp32 tensors at the boundary of the split path on the first forward of a weight set (engine.py).
__host__ __device__ inline void split_f32(float a, __half& hi, __half& lo) {
  a = fminf(fmaxf(a, -65504.0f), 65504.0f);
  hi = __float2half_rn(a);
  lo = __float2half_rn((a - __half2float(hi)) * kLoScale);
}
__host__ __device__ inline float join_f32(__half hi, __half lo) {
  return __half2float(hi) + __half2float(lo) * kLoInv;
}

// A split tensor: two fp16 planes with identical [pixel][channel] layout.
struct SplitPtr {
  __half* hi;
  __half* lo;
};

// ---- conv launch descriptor -------------------------------------------------------------------
enum Epilogue : int {
  EPI_ACT = 0,    // y = act(acc+bias) -> split planes d0 (and d1)
  EPI_ZR = 1,     // c<hidden: z=sigmoid -> f0 ; else r=sigmoid, r*h(f1) -> d0
  EPI_Q = 2,      // q=tanh ; h=(1-z)h+zq -> f1 and d0
  EPI_DELTA = 3,  // c<2: coords1(f1)[c] += v ; optional copy to f2
  EPI_F32 = 4     // f0[pix*cout+c] = scale*v
};
enum Act : int { ACT_NONE = 0, ACT_RELU = 1 };

struct ConvParams {
  // input activation (split planes), `in_stride` channels per pixel, first channel at in_choff
  const __half* in_hi;
  const __half* in_lo;
  int in_stride, in_choff;
  int cin_pad;  // channels per tap in the packed weights (multiple of 64)
  // Input VIEW (all 0 = the stride-1 'same' conv over a [B][h][w][in_stride] tensor).  The encoders use it for
  //  * strided convs: output pixel (oy, ox), tap (ky, kx) reads input (oy*sy + ky - pad_y, ox*sx + kx - pad_x) of an
  //    in_h x in_w input (TF SAME: pad before = total/2), out of range = 0 -- TMA element strides, no gather pass;
  //  * the 7x7 stride-2 stem as a 4x1 conv over a space-to-depth image whose view pixel spans in_cext = 64 channels =
  //    4 neighbouring physical pixels of in_stride = 16 channels (overlapping windows, encoder.cu).
  int in_w, in_h;       // spatial extent of the view (0: w, h)
  int in_rowpitch;      // elements between view rows (0: in_stride * in_w); images are in_rowpitch * in_h apart
  int in_cext;          // channels addressable from one view pixel (0: in_stride)
  int sx, sy;           // conv stride (0: 1)
  int pad_explicit, pad_x, pad_y;  // pad before, when not the symmetric (k-1)/2
  // K sub-range: only the 64-channel chunks i in [0, ck_count) are multiplied, chunk i -> channel chunk
  // ck(i) = ck_begin + i + (i >= ck_skip_at ? ck_skip : 0).  ck_count == 0 means "all chunks".
  // (The iteration-invariant `inp` slice of the GRU inputs is convolved once per pair and skipped afterwards.)
  int ck_begin, ck_count, ck_skip_at, ck_skip;
  const float* addend;  // optional fp32 [pixel][cout] added to the accumulator before bias/activation
  const float* flow_tail;  // EPI_ACT, 16-channel epilogue: coords1; the last two channels are written as flow = coords1 - grid
  double* stat_part;  // EPI_F32 + tensor-core wide epilogue: per-(sample, strip, channel) sum / sum of squares of the
  int stat_strips;    // stored values, [B][strips][2][cout] (strip = 4 * tile-in-image + lane quarter); encoder.cu
  int stash;      // 1: single-tile CTAs park the gate epilogues' fp32 operands in spare TMEM columns during the MMA loop
  int split_k;    // 1: K summed as (first half of the chunks) + (second half) (conv_tc.cu; cout <= 2, EPI_DELTA) ...
  int split_close;    // launcher: closing cluster barrier of the split-K pair (RAFT_B200_SPLITK_CLOSING_BARRIER, sanitizer runs)
  int split_cluster;  // ... set by the launcher: the halves run on the two CTAs of a cluster (one wave of pairs, batch 1)
  int cta_limit;  // > 0: at most this many persistent CTAs (a conv that runs beside another one on a forked stream)
  long long* dbg;       // optional phase timestamps (globaltimer ns), 8 slots per CTA; see tools/phase_times.py
  // packed weights [cout_pad][kh*kw][cin_pad] (K-major) as split planes + fp32 bias
  const __half* w_hi;
  const __half* w_lo;
  const float* bias;
  int cout, cout_pad, kh, kw;
  int w_per_batch;  // 1: the "weight" operand differs per batch element (correlation GEMM: fmap2)
  int B, h, w;
  // epilogue
  int epi, act, hidden;
  float scale;
  float div;  // EPI_F32: if non-zero, y = v / div instead of scale * v
  __half* d0_hi;
  __half* d0_lo;
  int d0_stride, d0_choff;
  __half* d1_hi;
  __half* d1_lo;
  int d1_stride, d1_choff;
  float* f0;
  float* f1;
  float* f2;
  // EPI_ACT: optional residual (split planes, res_stride channels per pixel): y = relu(res + act(acc + bias)), the block
  // output of ResidualBlock / BottleneckBlock (model_utils.py:31-35, 52-57)
  const __half* res_hi;
  const __half* res_lo;
  int res_stride;
};
__host__ __device__ inline int conv_sx(const ConvParams& p) { return p.sx > 0 ? p.sx : 1; }
__host__ __device__ inline int conv_sy(const ConvParams& p) { return p.sy > 0 ? p.sy : 1; }
__host__ __device__ inline int conv_pad_x(const ConvParams& p) { return p.pad_explicit ? p.pad_x : (p.kw - 1) / 2; }
__host__ __device__ inline int conv_pad_y(const ConvParams& p) { return p.pad_explicit ? p.pad_y : (p.kh - 1) / 2; }
__host__ __device__ inline int conv_in_w(const ConvParams& p) { return p.in_w > 0 ? p.in_w : p.w; }
__host__ __device__ inline int conv_in_h(const ConvParams& p) { return p.in_h > 0 ? p.in_h : p.h; }
__host__ __device__ inline int conv_rowpitch(const ConvParams& p) { return p.in_rowpitch > 0 ? p.in_rowpitch : p.in_stride * conv_in_w(p); }

// Gate non-linearities on the SFU: exp via ex2.approx (abs. error of the gate < 3e-7 for |x| < 16, i.e.
// below the 2^-22 operand truncation of the split GEMM that feeds them), reciprocal via rcp.approx.
// r01 profile: with libm expf/tanhf + IEEE division the GRU epilogues took as long as their MMA loops.
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_fast(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sigmoid_f(float x) { return rcp_fast(1.0f + ex2_fast(-1.4426950408889634f * x)); }
__device__ __forceinline__ float tanh_f(float x) {  // 1 - 2/(1+e^{2x}); exact limits at +-inf
  return fmaf(-2.0f, rcp_fast(1.0f + ex2_fast(2.8853900817779268f * x)), 1.0f);
}

// 256-bit global accesses (sm_100: LDG.256 / STG.256).  The tensor-core epilogues have one pixel per lane, so every lane
// of a warp-wide access touches a different 32-byte sector: 256-bit accesses fill the sector a lane touches instead of
// half of it and halve the number of LSU transactions of the epilogue (profiles/r01_notes.md).  32-byte aligned.
__device__ __forceinline__ void ld256(const float* src, float* d) {
  asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3]), "=f"(d[4]), "=f"(d[5]), "=f"(d[6]), "=f"(d[7])
               : "l"(src) : "memory");
}
__device__ __forceinline__ void ld256_nc(const float* src, float* d) {
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3]), "=f"(d[4]), "=f"(d[5]), "=f"(d[6]), "=f"(d[7])
               : "l"(src));
}
__device__ __forceinline__ void st256(float* dst, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "l"(dst), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}
__device__ __forceinline__ void st256_b32(void* dst, const uint32_t* v) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "l"(dst), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
// All destinations / operands of the conv are 32-byte aligned at 16-channel granularity (uniform per launch).
__device__ __forceinline__ bool epilogue_wide_ok(const ConvParams& p) {
  auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 31) == 0; };
  bool ok = (p.cout & 15) == 0 && al(p.bias) && al(p.addend) && al(p.d0_hi) && al(p.d0_lo) && al(p.d1_hi) && al(p.d1_lo) &&
            al(p.f0) && al(p.f1);
  if (p.epi == EPI_ACT) {
    ok = ok && ((p.d0_stride | p.d0_choff) & 15) == 0;
    if (p.res_hi) ok = ok && al(p.res_hi) && al(p.res_lo) && (p.res_stride & 15) == 0;
    if (p.d1_hi) ok = ok && ((p.d1_stride | p.d1_choff) & 15) == 0;
  } else if (p.epi == EPI_ZR || p.epi == EPI_Q) {
    ok = ok && ((p.d0_stride | p.d0_choff) & 15) == 0 && (p.hidden & 15) == 0;
  } else if (p.epi == EPI_DELTA) {
    ok = false;
  }
  return ok;
}

// Store NV consecutive output channels [c, c+NV) of pixel `pix`; v holds acc (bias not yet added).
// c is a multiple of NV; channel offsets of every destination are multiples of 8.
template <int NV>
__device__ __forceinline__ void epilogue_store(const ConvParams& p, int pix, int c, const float* v) {
  if (c >= p.cout) return;
  float y[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) y[i] = v[i] + ((p.bias && c + i < p.cout) ? __ldg(p.bias + c + i) : 0.f);
  const bool full = (c + NV <= p.cout);
  if (p.addend) {
    const float* ad = p.addend + (size_t)pix * p.cout + c;
    if (full && NV % 4 == 0 && (p.cout & 3) == 0) {
#pragma unroll
      for (int i = 0; i < NV; i += 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(ad + i));
        y[i] += t.x; y[i + 1] += t.y; y[i + 2] += t.z; y[i + 3] += t.w;
      }
    } else {
      for (int i = 0; i < NV; ++i)
        if (c + i < p.cout) y[i] += __ldg(ad + i);
    }
  }

  auto load_f32 = [&](const float* src, float* dst) {  // NV consecutive floats, 4*NV-byte aligned
    if constexpr (NV % 4 == 0) {
#pragma unroll
      for (int i = 0; i < NV; i += 4) {
        const float4 t = *reinterpret_cast<const float4*>(src + i);
        dst[i] = t.x; dst[i + 1] = t.y; dst[i + 2] = t.z; dst[i + 3] = t.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < NV; ++i) dst[i] = src[i];
    }
  };
  auto store_f32 = [&](float* dst, const float* src) {
    if constexpr (NV % 4 == 0) {
#pragma unroll
      for (int i = 0; i < NV; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(src[i], src[i + 1], src[i + 2], src[i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < NV; ++i) dst[i] = src[i];
    }
  };
  auto store_split = [&](__half* dhi, __half* dlo, int stride, int choff, int cc, const float* val) {
    size_t off = (size_t)pix * stride + choff + cc;
    if (full) {
      __align__(16) __half h[NV];
      __align__(16) __half l[NV];
#pragma unroll
      for (int i = 0; i < NV; ++i) split_f32(val[i], h[i], l[i]);
      if constexpr (NV == 8) {
        *reinterpret_cast<uint4*>(dhi + off) = *reinterpret_cast<const uint4*>(h);
        *reinterpret_cast<uint4*>(dlo + off) = *reinterpret_cast<const uint4*>(l);
      } else if constexpr (NV == 4) {
        *reinterpret_cast<uint2*>(dhi + off) = *reinterpret_cast<const uint2*>(h);
        *reinterpret_cast<uint2*>(dlo + off) = *reinterpret_cast<const uint2*>(l);
      } else {
#pragma unroll
        for (int i = 0; i < NV; ++i) { dhi[off + i] = h[i]; dlo[off + i] = l[i]; }
      }
    } else {
      for (int i = 0; i < NV; ++i)
        if (c + i < p.cout) {
          __half h, l;
          split_f32(val[i], h, l);
          dhi[off + i] = h;
          dlo[off + i] = l;
        }
    }
  };

  switch (p.epi) {
    case EPI_ACT: {
      if (p.act == ACT_RELU) {
#pragma unroll
        for (int i = 0; i < NV; ++i) y[i] = fmaxf(y[i], 0.f);
      }
      if (p.res_hi) {
        const size_t ro = (size_t)pix * p.res_stride + c;
        for (int i = 0; i < NV; ++i)
          if (c + i < p.cout) y[i] = fmaxf(join_f32(p.res_hi[ro + i], p.res_lo[ro + i]) + y[i], 0.f);
      }
      store_split(p.d0_hi, p.d0_lo, p.d0_stride, p.d0_choff, c, y);
      if (p.d1_hi) store_split(p.d1_hi, p.d1_lo, p.d1_stride, p.d1_choff, c, y);
    } break;
    case EPI_ZR: {
      // hidden is a multiple of NV (96, 128) so a group never straddles z|r.  All loads are issued
      // before any store: f0/f1 may alias as far as the compiler knows, and interleaving them would
      // serialise one L2 round trip per channel.
      if (c < p.hidden) {
        float z[NV];
#pragma unroll
        for (int i = 0; i < NV; ++i) z[i] = sigmoid_f(y[i]);
        store_f32(p.f0 + (size_t)pix * p.hidden + c, z);
      } else {
        const int ch = c - p.hidden;
        float hprev[NV];
        load_f32(p.f1 + (size_t)pix * p.hidden + ch, hprev);
#pragma unroll
        for (int i = 0; i < NV; ++i) y[i] = sigmoid_f(y[i]) * hprev[i];
        store_split(p.d0_hi, p.d0_lo, p.d0_stride, p.d0_choff, ch, y);
      }
    } break;
    case EPI_Q: {
      float z[NV], hprev[NV];
      load_f32(p.f0 + (size_t)pix * p.hidden + c, z);
      load_f32(p.f1 + (size_t)pix * p.hidden + c, hprev);
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const float q = tanh_f(y[i]);
        y[i] = (1.0f - z[i]) * hprev[i] + z[i] * q;  // model_utils.py:147,155,168
      }
      store_f32(p.f1 + (size_t)pix * p.hidden + c, y);
      store_split(p.d0_hi, p.d0_lo, p.d0_stride, p.d0_choff, c, y);
    } break;
    case EPI_DELTA: {
      for (int i = 0; i < NV; ++i)
        if (c + i < 2) {
          size_t o = (size_t)pix * 2 + c + i;
          p.f1[o] = p.f1[o] + y[i];  // RAFT.py:102
          if (p.f2) p.f2[o] = y[i];
        }
    } break;
    case EPI_F32: {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        if (p.act == ACT_RELU) y[i] = fmaxf(y[i], 0.f);
        y[i] = (p.div != 0.f) ? y[i] / p.div : p.scale * y[i];
      }
      float* dst = p.f0 + (size_t)pix * p.cout + c;
      if (full && (p.cout & 3) == 0 && NV % 4 == 0) {
#pragma unroll
        for (int i = 0; i < NV; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(y[i], y[i + 1], y[i + 2], y[i + 3]);
      } else {
        for (int i = 0; i < NV; ++i)
          if (c + i < p.cout) dst[i] = y[i];
      }
    } break;
  }
}

// ---- lean 16-channel epilogue (tensor-core kernels, epilogue_wide_ok() launches) ----------------------------------
// Same arithmetic as epilogue_store<NV>, element for element; 256-bit global accesses, no per-element bounds logic.
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  a = fminf(fmaxf(a, -65504.0f), 65504.0f);  // saturate like split_f32
  b = fminf(fmaxf(b, -65504.0f), 65504.0f);
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn((a - hf.x) * kLoScale, (b - hf.y) * kLoScale);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void store_split16(__half* dhi, __half* dlo, size_t off, const float* y) {
  uint32_t h[8], l[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) split2(y[2 * i], y[2 * i + 1], h[i], l[i]);
  st256_b32(dhi + off, h);
  st256_b32(dlo + off, l);
}
__device__ __forceinline__ void load16(const float* src, float* d) {
  ld256(src, d);
  ld256(src + 8, d + 8);
}
__device__ __forceinline__ void store16(float* dst, const float* v) {
  st256(dst, v);
  st256(dst + 8, v + 8);
}
// ---- TMEM as a prefetch buffer for epilogue operands ("stash") -------------------------------------------------------
// At batch 1 a conv CTA owns ONE tile, so the second accumulator buffer in TMEM is never used by the MMA warp.  The 16
// epilogue warps idle during the MMA loop; they load the fp32 operands the gate epilogues need (hoisted addend, z, h) and
// park them there with tcgen05.st -- after the loop the epilogue reads them back next to the accumulators (tcgen05.ld,
// tens of cycles) instead of paying two dependent L2 round trips per 16-channel chunk with only 4 warps per scheduler
// to hide them (r01 what-if: the epilogue's global loads cost 13 us per update step).  Holding them in registers instead
// was tried in round 1 and spilled (96-register cap).  Layout: operand k of tile column c at TMEM column stash + k*BN + c.
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]),
        "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// load + wait in one asm block: the registers are valid when it returns
__device__ __forceinline__ void tmem_ld16_sync(uint32_t taddr, float* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]), "=f"(v[9]),
        "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
      : "r"(taddr)
      : "memory");
}
struct Stash {
  uint32_t taddr;  // TMEM address (lane quarter of this warp, first stash column) or 0 = operands come from global memory
  int bn;          // tile width = column distance between stashed operands
  int cl;          // column of the current 16-channel chunk inside the tile
};

// `live` = this lane's pixel exists.  Without a stash the caller only calls live lanes; WITH a stash every lane of the warp
// must come here (tcgen05.ld is .sync.aligned: warp-collective) and dead lanes skip the global accesses.
__device__ __forceinline__ void epilogue_wide16(const ConvParams& p, int pix, int c, float* y, const Stash st = Stash{0, 0, 0},
                                                const bool live = true) {
  if (p.bias) {
    float t[16];
    ld256_nc(p.bias + c, t);
    ld256_nc(p.bias + c + 8, t + 8);
#pragma unroll
    for (int i = 0; i < 16; ++i) y[i] += t[i];
  }
  if (p.addend) {
    float t[16];
    const float* ad = p.addend + (size_t)pix * p.cout + c;
    if (st.taddr) {
      tmem_ld16_sync(st.taddr + st.cl, t);
    } else {
      ld256_nc(ad, t);
      ld256_nc(ad + 8, t + 8);
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) y[i] += t[i];
  }
  switch (p.epi) {
    case EPI_ACT: {
      if (p.act == ACT_RELU) {
#pragma unroll
        for (int i = 0; i < 16; ++i) y[i] = fmaxf(y[i], 0.f);
      }
      if (p.res_hi) {  // block output: relu(x + y), x as split planes (16 channels = 32 bytes per plane)
        __align__(32) __half rh[16], rl[16];
        const size_t ro = (size_t)pix * p.res_stride + c;
        ld256_nc(reinterpret_cast<const float*>(p.res_hi + ro), reinterpret_cast<float*>(rh));
        ld256_nc(reinterpret_cast<const float*>(p.res_lo + ro), reinterpret_cast<float*>(rl));
#pragma unroll
        for (int i = 0; i < 16; ++i) y[i] = fmaxf(join_f32(rh[i], rl[i]) + y[i], 0.f);
      }
      if (p.flow_tail && c + 16 == p.cout) {
        // motion encoder: [126 conv channels | flow] (model_utils.py:119) -- the flow slot completes the 16-channel group,
        // same arithmetic as flow_conv7_kernel (coords1 - coords_grid, RAFT.py:95)
        const int x = pix % p.w, yy = (pix / p.w) % p.h;
        const float2 cc = *reinterpret_cast<const float2*>(p.flow_tail + (size_t)pix * 2);
        y[14] = cc.x - (float)x;
        y[15] = cc.y - (float)yy;
      }
      store_split16(p.d0_hi, p.d0_lo, (size_t)pix * p.d0_stride + p.d0_choff + c, y);
      if (p.d1_hi) store_split16(p.d1_hi, p.d1_lo, (size_t)pix * p.d1_stride + p.d1_choff + c, y);
    } break;
    case EPI_ZR: {
      if (c < p.hidden) {
#pragma unroll
        for (int i = 0; i < 16; ++i) y[i] = sigmoid_f(y[i]);
        if (live) store16(p.f0 + (size_t)pix * p.hidden + c, y);
      } else {
        const int ch = c - p.hidden;
        float hprev[16];
        if (st.taddr) tmem_ld16_sync(st.taddr + st.bn + st.cl, hprev);
        else load16(p.f1 + (size_t)pix * p.hidden + ch, hprev);
#pragma unroll
        for (int i = 0; i < 16; ++i) y[i] = sigmoid_f(y[i]) * hprev[i];
        if (live) store_split16(p.d0_hi, p.d0_lo, (size_t)pix * p.d0_stride + p.d0_choff + ch, y);
      }
    } break;
    case EPI_Q: {
      float z[16], hprev[16];
      float* hp = p.f1 + (size_t)pix * p.hidden + c;
      if (st.taddr) {
        tmem_ld16_sync(st.taddr + st.bn + st.cl, z);
        tmem_ld16_sync(st.taddr + 2 * st.bn + st.cl, hprev);
      } else {
        load16(p.f0 + (size_t)pix * p.hidden + c, z);
        load16(hp, hprev);
      }
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float q = tanh_f(y[i]);
        y[i] = (1.0f - z[i]) * hprev[i] + z[i] * q;  // model_utils.py:147,155,168
      }
      if (live) {
        store16(hp, y);
        store_split16(p.d0_hi, p.d0_lo, (size_t)pix * p.d0_stride + p.d0_choff + c, y);
      }
    } break;
    default: {  // EPI_F32
      if (p.act == ACT_RELU) {
#pragma unroll
        for (int i = 0; i < 16; ++i) y[i] = fmaxf(y[i], 0.f);
      }
      if (p.div != 0.f) {
#pragma unroll
        for (int i = 0; i < 16; ++i) y[i] = y[i] / p.div;
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) y[i] = p.scale * y[i];
      }
      store16(p.f0 + (size_t)pix * p.cout + c, y);
    } break;
  }
}

// Per-channel sum and sum of squares over the 32 pixels (lanes) of a warp for the 16 channels each lane holds
// (instance-norm statistics fused into the conv epilogue).  Recursive halving: after the xor-16/8/4/2 exchanges lane l
// owns channel 8*b4 + 4*b3 + 2*b2 + b1 (b_i = bit i of l), the xor-1 step completes the sum; 32 shuffles, fixed order.
__device__ __forceinline__ void warp_stats16(const float* y, float& s, float& s2, int& ch) {
  const unsigned lane = threadIdx.x & 31u;
  float a[8], b[8];
  {
    const bool up = (lane & 16u) != 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float keep = up ? y[i + 8] : y[i], send = up ? y[i] : y[i + 8];
      a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
      b[i] = keep * keep + __shfl_xor_sync(0xffffffffu, send * send, 16);
    }
  }
#pragma unroll
  for (int w = 4; w >= 1; w >>= 1) {  // 8 -> 4 -> 2 -> 1 values per lane, partner at xor 2w
    const bool up = (lane & (unsigned)(2 * w)) != 0;
#pragma unroll
    for (int i = 0; i < w; ++i) {
      const float ka = up ? a[i + w] : a[i], sa = up ? a[i] : a[i + w];
      const float kb = up ? b[i + w] : b[i], sb = up ? b[i] : b[i + w];
      a[i] = ka + __shfl_xor_sync(0xffffffffu, sa, 2 * w);
      b[i] = kb + __shfl_xor_sync(0xffffffffu, sb, 2 * w);
    }
  }
  s = a[0] + __shfl_xor_sync(0xffffffffu, a[0], 1);
  s2 = b[0] + __shfl_xor_sync(0xffffffffu, b[0], 1);
  ch = (int)(((lane >> 4) & 1u) * 8u + ((lane >> 3) & 1u) * 4u + ((lane >> 2) & 1u) * 2u + ((lane >> 1) & 1u));
}

// back ends
int launch_conv_simt(const ConvParams& p, cudaStream_t s);
int launch_conv_tc(const ConvParams& p, cudaStream_t s);
int conv_tc_tiles_per_image(int h, int w);
bool conv_tc_fused_stats_ok(const ConvParams& p);
inline int launch_conv(const ConvParams& p, cudaStream_t s) {
  return math_mode() == RB_MATH_SIMT ? launch_conv_simt(p, s) : launch_conv_tc(p, s);
}

__device__ __forceinline__ long long gtime_ns() {
  long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t) :: "memory");  // "memory": keeps the read on its side of barriers
  return t;
}
inline int level_dim(int d, int level) { return d >> level; }
__host__ __device__ inline int conv_chunks(const ConvParams& p) { return p.ck_count > 0 ? p.ck_count : p.cin_pad / 64; }
__host__ __device__ inline int conv_chunk(const ConvParams& p, int i) {
  return p.ck_count > 0 ? p.ck_begin + i + (i >= p.ck_skip_at ? p.ck_skip : 0) : i;
}

}  // namespace rb
