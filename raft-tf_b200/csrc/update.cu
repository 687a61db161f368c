// A5-A12: motion encoder, (Sep)ConvGRU, flow head, mask head and the iteration loop.
// Reference: networks/model_utils.py:110-194, networks/RAFT.py:84-102.
//
// Data layout (per frame-pair batch, npix = B*h*w; every activation is a split fp16 tensor
// [npix][C] = hi plane followed by lo plane, see common.cuh):
//   CORR [Ccorr]  lookup output, 4*(2r+1)^2 channels zero-padded to a multiple of 64
//   C1   [256]    relu(convc1)                                   (things only)
//   CF   [cf]     [cor | flo]      = input of encoder/conv       (model_utils.py:117,127)
//   F1   [f1]     relu(convf1)
//   FL   [8]      the flow as a zero-padded image [B][h][w+8] (channels 0,1): operand of convf1's 8-pixel window view
//   HX   [hx]     [h | inp | motion_out | flow | 0-pad] = GRU z/r input (cat_hx, :141,150,160)
//   QX   [hx]     [r*h | inp | motion_out | flow | 0-pad] = GRU q input (:144,153,165)
//   FH   [fh]     relu(flow_head/conv1); reused for relu(mask/0)
//   H, Z fp32 [hidden]  recurrent state and the update gate
// Concatenations are never materialised: producers write at channel offsets of HX/QX/CF.
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "tc_common.cuh"

namespace rb {

int launch_lookup(const float* pyramid, const float* coords, float* out_f32, __half* out_hi,
                  __half* out_lo, int out_stride, int B, int h, int w, int radius, cudaStream_t s);
int launch_lookup_otf(const float* fmap1, const float* fmap2, const float* pooled, const float* coords, float* out_f32,
                      __half* out_hi, __half* out_lo, int out_stride, int B, int h, int w, int C, int radius, cudaStream_t s);

// ---------------------------------------------------------------------------------------------
// static description of the two variants
// ---------------------------------------------------------------------------------------------
struct RefConv {
  const char* name;
  int kh, kw, cin, cout;
};

static const RefConv kThingsConvs[] = {
    {"update_block/encoder/convc1", 1, 1, 324, 256}, {"update_block/encoder/convc2", 3, 3, 256, 192},
    {"update_block/encoder/convf1", 7, 7, 2, 128},   {"update_block/encoder/convf2", 3, 3, 128, 64},
    {"update_block/encoder/conv", 3, 3, 256, 126},   {"update_block/gru/convz1", 1, 5, 384, 128},
    {"update_block/gru/convr1", 1, 5, 384, 128},     {"update_block/gru/convq1", 1, 5, 384, 128},
    {"update_block/gru/convz2", 5, 1, 384, 128},     {"update_block/gru/convr2", 5, 1, 384, 128},
    {"update_block/gru/convq2", 5, 1, 384, 128},     {"update_block/flow_head/conv1", 3, 3, 128, 256},
    {"update_block/flow_head/conv2", 3, 3, 256, 2},  {"update_block/mask/0", 3, 3, 128, 256},
    {"update_block/mask/2", 1, 1, 256, 576}};
static const RefConv kSmallConvs[] = {
    {"update_block/encoder/convc1", 1, 1, 196, 96}, {"update_block/encoder/convf1", 7, 7, 2, 64},
    {"update_block/encoder/convf2", 3, 3, 64, 32},  {"update_block/encoder/conv", 3, 3, 128, 80},
    {"update_block/gru/convz", 3, 3, 242, 96},      {"update_block/gru/convr", 3, 3, 242, 96},
    {"update_block/gru/convq", 3, 3, 242, 96},      {"update_block/flow_head/conv1", 3, 3, 96, 128},
    {"update_block/flow_head/conv2", 3, 3, 128, 2}};

// packed (device) convs; src = indices into the reference list (two for the merged z|r conv)
enum PackedId {
  P_CONVC1 = 0, P_CONVC2, P_CONVF2, P_MOTION, P_ZR1, P_Q1, P_ZR2, P_Q2, P_FH1, P_FH2, P_MASK0, P_MASK2, P_COUNT
};
struct PackedConv {
  int src0, src1;  // reference conv indices (-1 = none)
  int cin_pad;
};

struct Variant {
  int small, hidden, ctx, radius, corr_ch, corr_pad, c1, cf, cor, f1, hx, fh, mo_out, nref;
  const RefConv* ref;
  int convf1_ref;
  PackedConv pk[P_COUNT];
};

static const Variant kThings = {
    0, 128, 128, 4, 324, 384, 256, 256, 192, 128, 384, 256, 126, 15, kThingsConvs, 2,
    {{0, -1, 384}, {1, -1, 256}, {3, -1, 128}, {4, -1, 256}, {5, 6, 384}, {7, -1, 384}, {8, 9, 384},
     {10, -1, 384}, {11, -1, 128}, {12, -1, 256}, {13, -1, 128}, {14, -1, 256}}};
static const Variant kSmall = {
    1, 96, 64, 3, 196, 256, 0, 128, 96, 64, 256, 128, 80, 9, kSmallConvs, 1,
    {{0, -1, 256}, {-1, -1, 0}, {2, -1, 64}, {3, -1, 128}, {4, 5, 256}, {6, -1, 256}, {-1, -1, 0},
     {-1, -1, 0}, {7, -1, 128}, {8, -1, 128}, {-1, -1, 0}, {-1, -1, 0}}};

static inline const Variant& variant(int small) { return small ? kSmall : kThings; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int pad16(int c) { return (c + 15) / 16 * 16; }

// ---- packed weight blob -------------------------------------------------------------------------
struct PackedLayout {
  size_t hi[P_COUNT], lo[P_COUNT], bias[P_COUNT];  // byte offsets
  int cout[P_COUNT], cout_pad[P_COUNT], kh[P_COUNT], kw[P_COUNT];
  size_t f1_w, f1_b;  // convf1: fp32 [49*2][cout] and bias (CUDA-core kernel)
  size_t f1t_hi, f1t_lo, f1t_bias;  // convf1 for the tensor-core path: 7x1 conv over the 8-pixel window view, [cout_pad][7][64]
  int f1t_cout, f1t_cout_pad;
  size_t total;
};

static PackedLayout packed_layout(const Variant& v) {
  PackedLayout L;
  memset(&L, 0, sizeof(L));
  size_t off = 0;
  for (int i = 0; i < P_COUNT; ++i) {
    const PackedConv& pc = v.pk[i];
    if (pc.src0 < 0) continue;
    const RefConv& r0 = v.ref[pc.src0];
    int cout = r0.cout + (pc.src1 >= 0 ? v.ref[pc.src1].cout : 0);
    L.cout[i] = cout;
    L.cout_pad[i] = pad16(cout);
    L.kh[i] = r0.kh;
    L.kw[i] = r0.kw;
    size_t plane = (size_t)L.cout_pad[i] * r0.kh * r0.kw * pc.cin_pad * sizeof(__half);
    L.hi[i] = off; off = align_up(off + plane, 256);
    L.lo[i] = off; off = align_up(off + plane, 256);
    L.bias[i] = off; off = align_up(off + (size_t)L.cout_pad[i] * sizeof(float), 256);
  }
  const RefConv& f = v.ref[v.convf1_ref];
  L.f1_w = off; off = align_up(off + (size_t)f.kh * f.kw * f.cin * f.cout * sizeof(float), 256);
  L.f1_b = off; off = align_up(off + (size_t)f.cout * sizeof(float), 256);
  L.f1t_cout = f.cout; L.f1t_cout_pad = pad16(f.cout);
  {
    const size_t plane = (size_t)L.f1t_cout_pad * 7 * 64 * sizeof(__half);
    L.f1t_hi = off; off = align_up(off + plane, 256);
    L.f1t_lo = off; off = align_up(off + plane, 256);
    L.f1t_bias = off; off = align_up(off + (size_t)L.f1t_cout_pad * sizeof(float), 256);
  }
  L.total = off;
  return L;
}

// ---- activation workspace -------------------------------------------------------------------------
struct Workspace {
  SplitPtr corr, c1, cf, f1, hx, qx, fh;
  SplitPtr fl;  // flow as split planes [B][h][w + 8][8]: 3 zero pixels left, 5 right, channels 0,1 = flow (convf1's window view)
  float* H;
  float* Z;
  float* pre[4];  // things: bias + conv over the `inp` channels of zr1, q1, zr2, q2 (iteration-invariant)
  size_t total;
};

static Workspace workspace_layout(const Variant& v, size_t npix, void* base) {
  Workspace W;
  char* b = reinterpret_cast<char*>(base);
  size_t off = 0;
  auto split = [&](int C) {
    SplitPtr sp;
    size_t plane = align_up(npix * (size_t)C * sizeof(__half), 1024);
    sp.hi = reinterpret_cast<__half*>(b + off);
    sp.lo = reinterpret_cast<__half*>(b + off + plane);
    off += 2 * plane;
    return sp;
  };
  W.corr = split(v.corr_pad);
  W.c1 = split(v.c1 > 0 ? v.c1 : 64);
  W.cf = split(v.cf);
  W.f1 = split(v.f1);
  W.hx = split(v.hx);
  W.qx = split(v.hx);
  W.fh = split(v.fh);
  {  // (w + 8) <= 2 w for every admissible grid (w >= 8): 2 * npix pixels of 8 channels bound the padded flow image
    const size_t plane = align_up(2 * npix * 8 * sizeof(__half), 1024);
    W.fl.hi = reinterpret_cast<__half*>(b + off);
    W.fl.lo = reinterpret_cast<__half*>(b + off + plane);
    off += 2 * plane;
  }
  size_t fsz = align_up(npix * (size_t)v.hidden * sizeof(float), 1024);
  W.H = reinterpret_cast<float*>(b + off); off += fsz;
  W.Z = reinterpret_cast<float*>(b + off); off += fsz;
  for (int i = 0; i < 4; ++i) {
    W.pre[i] = nullptr;
    if (!v.small) {
      W.pre[i] = reinterpret_cast<float*>(b + off);
      off += align_up(npix * (size_t)((i & 1) ? v.hidden : 2 * v.hidden) * sizeof(float), 1024);
    }
  }
  W.total = off;
  return W;
}

// ---------------------------------------------------------------------------------------------
// small kernels
// ---------------------------------------------------------------------------------------------
__global__ void set_state_kernel(const float* __restrict__ net, const float* __restrict__ inp, Workspace W,
                                 int npix, int hidden, int ctx, int hx) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  int per = hidden + ctx;
  if (i >= (size_t)npix * per) return;
  int pix = i / per, c = i % per;
  __half hi, lo;
  if (c < hidden) {
    float v = net[(size_t)pix * hidden + c];
    W.H[(size_t)pix * hidden + c] = v;
    split_f32(v, hi, lo);
    W.hx.hi[(size_t)pix * hx + c] = hi;
    W.hx.lo[(size_t)pix * hx + c] = lo;
  } else {
    float v = inp[(size_t)pix * ctx + (c - hidden)];
    split_f32(v, hi, lo);
    size_t o = (size_t)pix * hx + c;
    W.hx.hi[o] = hi; W.hx.lo[o] = lo;
    W.qx.hi[o] = hi; W.qx.lo[o] = lo;
  }
}

// net = tanh(cnet[..., :hidden]), inp = relu(cnet[..., hidden:])  (RAFT.py:85-87)
__global__ void set_state_cnet_kernel(const float* __restrict__ cnet, Workspace W, int npix, int hidden, int ctx, int hx) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  int per = hidden + ctx;
  if (i >= (size_t)npix * per) return;
  int pix = i / per, c = i % per;
  float v = cnet[i];
  __half hi, lo;
  size_t o = (size_t)pix * hx + c;
  if (c < hidden) {
    v = tanhf(v);
    W.H[(size_t)pix * hidden + c] = v;
    split_f32(v, hi, lo);
    W.hx.hi[o] = hi; W.hx.lo[o] = lo;
  } else {
    v = fmaxf(v, 0.f);
    split_f32(v, hi, lo);
    W.hx.hi[o] = hi; W.hx.lo[o] = lo;
    W.qx.hi[o] = hi; W.qx.lo[o] = lo;
  }
}

__global__ void set_corr_kernel(const float* __restrict__ corr, SplitPtr dst, int npix, int ch, int stride) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)npix * ch) return;
  int pix = i / ch, c = i % ch;
  __half hi, lo;
  split_f32(corr[i], hi, lo);
  dst.hi[(size_t)pix * stride + c] = hi;
  dst.lo[(size_t)pix * stride + c] = lo;
}

__global__ void copy_f32_kernel(const float* __restrict__ src, float* __restrict__ dst, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

// encoder/convf1: 7x7 conv over the 2-channel flow + ReLU (model_utils.py:114,124), CUDA-core form: the cross-check back end
// (RB_MATH_SIMT), and grids narrower than the 8-pixel window of the tensor-core form (flow_prep_kernel below + conv_tc).
// flow = coords1 - coords_grid (RAFT.py:95) is formed while staging; SAME padding zero-pads the FLOW.  One thread per output channel, SEG-pixel row segment
// per block (SEG = 16 at batch 1: 440 blocks instead of 220 -- the kernel is latency-bound, and with the convf2 that
// follows it on the forked stream it must not finish later than lookup -> convc1 -> convc2 on the main stream); the flow itself is also written into the [.., flow] slot of HX/QX (concat_out, :119).
template <int COUT, int SEG>
__global__ void __launch_bounds__(COUT) flow_conv7_kernel(const float2* __restrict__ coords1,
                                                          const float* __restrict__ Wf,  // [98][COUT]
                                                          const float* __restrict__ bf, SplitPtr f1,
                                                          int f1_stride, SplitPtr hx, SplitPtr qx,
                                                          int hx_stride, int flow_choff, int h, int w) {
  __shared__ float2 patch[7][SEG + 6];
  const int x0 = blockIdx.x * SEG, y = blockIdx.y, b = blockIdx.z;
  const int c = threadIdx.x;
  for (int e = threadIdx.x; e < 7 * (SEG + 6); e += COUT) {
    int py = e / (SEG + 6), px = e % (SEG + 6);
    int sy = y + py - 3, sx = x0 + px - 3;
    float2 f = make_float2(0.f, 0.f);
    if (sy >= 0 && sy < h && sx >= 0 && sx < w) {
      float2 cc = coords1[(size_t)(b * h + sy) * w + sx];
      f = make_float2(cc.x - (float)sx, cc.y - (float)sy);
    }
    patch[py][px] = f;
  }
  float wr[98];
#pragma unroll
  for (int k = 0; k < 98; ++k) wr[k] = Wf[k * COUT + c];
  const float bias = bf[c];
  __syncthreads();
  for (int px = 0; px < SEG; ++px) {
    int x = x0 + px;
    if (x >= w) break;
    float acc = 0.f;
#pragma unroll
    for (int ky = 0; ky < 7; ++ky)
#pragma unroll
      for (int kx = 0; kx < 7; ++kx) {
        float2 f = patch[ky][px + kx];
        acc = fmaf(wr[(ky * 7 + kx) * 2 + 0], f.x, acc);
        acc = fmaf(wr[(ky * 7 + kx) * 2 + 1], f.y, acc);
      }
    acc = fmaxf(acc + bias, 0.f);
    size_t pix = (size_t)(b * h + y) * w + x;
    __half hi, lo;
    split_f32(acc, hi, lo);
    f1.hi[pix * f1_stride + c] = hi;
    f1.lo[pix * f1_stride + c] = lo;
    if (c < 2) {
      float2 f = patch[3][px + 3];
      split_f32(c == 0 ? f.x : f.y, hi, lo);
      size_t o = pix * hx_stride + flow_choff + c;
      hx.hi[o] = hi; hx.lo[o] = lo;
      qx.hi[o] = hi; qx.lo[o] = lo;
    }
  }
}

// Tensor-core convf1: the 7x7x2 conv as a 7x1 conv over a view whose pixel is a window of 8 neighbouring flow pixels x 8
// channels = 64 contiguous fp16 (the overlapping-window view of the encoder stem, ConvParams in common.cuh): K = 7 x 64 of
// which 98 are non-zero -- 7 k-iterations on the tensor cores instead of 12 544 FMA per pixel on the CUDA cores, whose blocks
// cannot share an SM with a conv CTA (what-if without the CUDA-core kernel: -5 us per update step at batch 1, -48 us at 8).
// This pass writes the padded flow image [B][h][w + 8][8] (pad pixels and channels 2..7 = 0, so no reliance on earlier
// contents) and the [.., flow] slots of HX / QX (concat_out, model_utils.py:119).  One thread per padded pixel.
__global__ void flow_prep_kernel(const float2* __restrict__ coords1, SplitPtr fl, SplitPtr hx, SplitPtr qx, int hx_stride,
                                 int flow_choff, int B, int h, int w) {
  const int Wp = w + 8;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * h * Wp) return;
  const int xp = i % Wp, y = (i / Wp) % h, b = i / ((size_t)Wp * h);
  const int x = xp - 3;
  uint4 vh = make_uint4(0, 0, 0, 0), vl = vh;
  if (x >= 0 && x < w) {
    const size_t pix = (size_t)(b * h + y) * w + x;
    const float2 cc = coords1[pix];
    __half h0, l0, h1, l1;
    split_f32(cc.x - (float)x, h0, l0);  // flow = coords1 - coords_grid (RAFT.py:95)
    split_f32(cc.y - (float)y, h1, l1);
    vh.x = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
    vl.x = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
    const size_t o = pix * hx_stride + flow_choff;
    *reinterpret_cast<uint32_t*>(hx.hi + o) = vh.x; *reinterpret_cast<uint32_t*>(hx.lo + o) = vl.x;
    *reinterpret_cast<uint32_t*>(qx.hi + o) = vh.x; *reinterpret_cast<uint32_t*>(qx.lo + o) = vl.x;
  }
  *reinterpret_cast<uint4*>(fl.hi + i * 8) = vh;
  *reinterpret_cast<uint4*>(fl.lo + i * 8) = vl;
}

// ---------------------------------------------------------------------------------------------
// one update-block application
// ---------------------------------------------------------------------------------------------
static ConvParams base_params(const Variant& v, const PackedLayout& L, const void* blob, int id, SplitPtr in,
                              int in_stride, int in_choff, int B, int h, int w) {
  ConvParams p;
  memset(&p, 0, sizeof(p));
  const char* bb = reinterpret_cast<const char*>(blob);
  p.in_hi = in.hi; p.in_lo = in.lo; p.in_stride = in_stride; p.in_choff = in_choff;
  p.cin_pad = v.pk[id].cin_pad;
  p.w_hi = reinterpret_cast<const __half*>(bb + L.hi[id]);
  p.w_lo = reinterpret_cast<const __half*>(bb + L.lo[id]);
  p.bias = reinterpret_cast<const float*>(bb + L.bias[id]);
  p.cout = L.cout[id]; p.cout_pad = L.cout_pad[id]; p.kh = L.kh[id]; p.kw = L.kw[id];
  p.B = B; p.h = h; p.w = w;
  p.hidden = v.hidden; p.scale = 1.f;
  return p;
}

// The `inp` slice of the GRU inputs ([h|inp|motion|flow], model_utils.py:141,144,150,153) never changes during
// the iterations of one pair (RAFT.py:85-87,97-101), so its contribution (and the bias) to the z|r and q
// convolutions is computed once in rb_update_set_state* and added in the epilogue: the per-iteration K loop
// skips those channels (-1/3 of the GRU MMA work and operand traffic; identical up to fp32 summation order).
// Only when the slice is aligned to the 64-channel chunks (raft-things: [128,256)).
static inline bool can_hoist(const Variant& v) {
  static const bool off = getenv("RAFT_B200_NO_HOIST") != nullptr;  // A/B knob
  return !off && !v.small && v.hidden % 64 == 0 && v.ctx % 64 == 0;
}
static void hoist_inp(const Variant& v, const Workspace& W, int idx, ConvParams& p) {
  if (!can_hoist(v)) return;
  const int total = v.hx / 64, inp0 = v.hidden / 64, ninp = v.ctx / 64;
  p.ck_begin = 0; p.ck_count = total - ninp; p.ck_skip_at = inp0; p.ck_skip = ninp;
  p.addend = W.pre[idx];
  p.bias = nullptr;  // folded into the addend
}

// Phase-timestamp debug buffer (tools/phase_times.py): rb_debug_set_buffer(ptr, convs) makes the next update
// step record 8 timestamps per CTA for each of its convs, in launch order, 4096 CTAs per conv.
static thread_local long long* g_dbg = nullptr;
static thread_local int g_dbg_idx = 0;
static int launch_conv_dbg(ConvParams& p, cudaStream_t s) {
  if (g_dbg) p.dbg = g_dbg + (size_t)(g_dbg_idx++) * 4096 * 8;
  return launch_conv(p, s);
}

static void set_act(ConvParams& p, int act, SplitPtr d0, int stride0, int choff0) {
  p.epi = EPI_ACT; p.act = act;
  p.d0_hi = d0.hi; p.d0_lo = d0.lo; p.d0_stride = stride0; p.d0_choff = choff0;
}

// Second stream for the flow branch of the motion encoder (convf1 -> convf2), which is independent of the
// correlation branch (lookup -> convc1 -> convc2) until encoder/conv joins them (model_utils.py:112-118).
// At batch 1 a conv uses 55-110 of the 148 SMs, so the two branches genuinely overlap.  Fork/join with
// events is also how the branch is expressed inside a CUDA-graph capture.
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  int device = -1;
};
static int side_stream(SideStream** out) {
  static thread_local SideStream per_dev[16];  // one set of streams / events per (calling thread, device ordinal)
  int dev = 0;
  RB_CHECK_CUDA(cudaGetDevice(&dev));
  RB_REQUIRE(dev >= 0 && dev < 16, RB_ERR_UNSUPPORTED, "device ordinal %d (the side streams are kept for ordinals 0..15)", dev);
  SideStream& ss = per_dev[dev];
  if (ss.device != dev) {
    RB_CHECK_CUDA(cudaStreamCreateWithFlags(&ss.stream, cudaStreamNonBlocking));
    RB_CHECK_CUDA(cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming));
    RB_CHECK_CUDA(cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming));
    ss.device = dev;
  }
  *out = &ss;
  return RB_OK;
}

// pyramid != nullptr: the lookup for this iteration is issued here too (on the main branch)
static int update_step(const Variant& v, const void* blob, void* wsp, float* coords1, float* delta_out,
                       float* mask_out, int B, int h, int w, cudaStream_t s, const float* pyramid = nullptr) {
  const size_t npix = (size_t)B * h * w;
  const PackedLayout L = packed_layout(v);
  const Workspace W = workspace_layout(v, npix, wsp);
  const char* bb = reinterpret_cast<const char*>(blob);
  const int xoff = v.hidden + v.ctx;      // channel offset of motion_out inside HX/QX
  const int foff = xoff + v.mo_out;       // channel offset of the raw flow
  int rc;
  g_dbg_idx = 0;
  // ---- motion encoder (model_utils.py:110-129) ----
  SideStream* ss;
  if ((rc = side_stream(&ss))) return rc;
  RB_CHECK_CUDA(cudaEventRecord(ss->fork, s));
  RB_CHECK_CUDA(cudaStreamWaitEvent(ss->stream, ss->fork, 0));
  {  // flow branch (side stream): convf1 (7x7) -> convf2
    const int seg = (long)B * h * w <= 16384 ? 16 : 32;  // same-box A/B at 55x128: 792 / 772 / 781 us per 4 iterations for 32 / 16 / 8
    const float* Wf = reinterpret_cast<const float*>(bb + L.f1_w);
    const float* bf = reinterpret_cast<const float*>(bb + L.f1_b);
    const float2* c1 = reinterpret_cast<const float2*>(coords1);
#define RB_LAUNCH_CONV7(COUT, SEG) \
    flow_conv7_kernel<COUT, SEG><<<dim3((w + SEG - 1) / SEG, h, B), COUT, 0, ss->stream>>>(c1, Wf, bf, W.f1, v.f1, W.hx, W.qx, v.hx, foff, h, w)
    // convf1 on the tensor cores (flow_prep_kernel + 7x1 conv over the window view); the CUDA-core math mode and grids
    // narrower than the window keep the CUDA-core kernel
    const bool f1_tc = math_mode() == RB_MATH_TC && (foff & 1) == 0 && (v.hx & 1) == 0 && w >= 8;
    if (f1_tc) {
      const size_t cells = (size_t)B * h * (w + 8);
      flow_prep_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, ss->stream>>>(c1, W.fl, W.hx, W.qx, v.hx, foff, B, h, w);
      RB_CHECK_LAUNCH("flow_prep_kernel");
      ConvParams p;
      memset(&p, 0, sizeof(p));
      p.in_hi = W.fl.hi; p.in_lo = W.fl.lo;
      p.in_stride = 8; p.in_cext = 64; p.in_w = w; p.in_h = h; p.in_rowpitch = (w + 8) * 8;
      p.cin_pad = 64; p.kh = 7; p.kw = 1;
      p.pad_explicit = 1; p.pad_x = 0; p.pad_y = 3;
      p.w_hi = reinterpret_cast<const __half*>(bb + L.f1t_hi);
      p.w_lo = reinterpret_cast<const __half*>(bb + L.f1t_lo);
      p.bias = reinterpret_cast<const float*>(bb + L.f1t_bias);
      p.cout = L.f1t_cout; p.cout_pad = L.f1t_cout_pad;
      p.B = B; p.h = h; p.w = w; p.hidden = v.hidden; p.scale = 1.f;
      set_act(p, ACT_RELU, W.f1, v.f1, 0);
      // batch 1: 28 CTAs = the 55 128-wide tiles in two full rounds (same-box sweep of both budgets, 4 iterations:
      // 19/38: 650, 28/28: 633, 28/38: 632, 38/38: 637, 55/38: 651, 38/55: 650, 110/38: 649 us)
      p.cta_limit = (long)B * h * w <= 16384 ? 28 : 0;
      if ((rc = launch_conv_dbg(p, ss->stream))) return rc;
    } else if (v.small) {
      if (seg == 16) RB_LAUNCH_CONV7(64, 16); else RB_LAUNCH_CONV7(64, 32);
    } else {
      if (seg == 16) RB_LAUNCH_CONV7(128, 16); else RB_LAUNCH_CONV7(128, 32);
    }
#undef RB_LAUNCH_CONV7
    RB_CHECK_LAUNCH("flow_conv7_kernel");
    {
      ConvParams p = base_params(v, L, blob, P_CONVF2, W.f1, v.f1, 0, B, h, w);
      set_act(p, ACT_RELU, W.cf, v.cf, v.cor);
      // convf2 runs beside convc1 / convc2 of the main stream: a small CTA budget keeps it off the SMs they need
      // (batch 1: the other convs use 110 of the 148 SMs; same-box A/B 770 -> 761 us per 4 iterations)
      p.cta_limit = (long)B * h * w <= 16384 ? 38 : 0;
      if ((rc = launch_conv_dbg(p, ss->stream))) return rc;
    }
    RB_CHECK_CUDA(cudaEventRecord(ss->join, ss->stream));
  }
  // correlation branch (main stream): [lookup ->] convc1 [-> convc2]
  if (pyramid) {
    if ((rc = launch_lookup(pyramid, coords1, nullptr, W.corr.hi, W.corr.lo, v.corr_pad, B, h, w, v.radius, s))) return rc;
  }
  if (!v.small) {
    ConvParams p = base_params(v, L, blob, P_CONVC1, W.corr, v.corr_pad, 0, B, h, w);
    set_act(p, ACT_RELU, W.c1, v.c1, 0);
    if ((rc = launch_conv_dbg(p, s))) return rc;
    p = base_params(v, L, blob, P_CONVC2, W.c1, v.c1, 0, B, h, w);
    set_act(p, ACT_RELU, W.cf, v.cf, 0);
    if ((rc = launch_conv_dbg(p, s))) return rc;
  } else {
    ConvParams p = base_params(v, L, blob, P_CONVC1, W.corr, v.corr_pad, 0, B, h, w);
    set_act(p, ACT_RELU, W.cf, v.cf, 0);
    if ((rc = launch_conv_dbg(p, s))) return rc;
  }
  RB_CHECK_CUDA(cudaStreamWaitEvent(s, ss->join, 0));
  {
    ConvParams p = base_params(v, L, blob, P_MOTION, W.cf, v.cf, 0, B, h, w);
    set_act(p, ACT_RELU, W.hx, v.hx, xoff);
    p.d1_hi = W.qx.hi; p.d1_lo = W.qx.lo; p.d1_stride = v.hx; p.d1_choff = xoff;
    if (math_mode() == RB_MATH_TC && (p.cout & 15) == 14 && p.cout + 2 <= p.cout_pad && foff == xoff + p.cout) {
      // things: 126 channels + the 2 flow channels right behind them = one full 16-channel group -> the tensor-core
      // epilogue writes the flow slot too and takes its 256-bit path (the weight rows / biases 126,127 are zero)
      p.cout += 2;
      p.flow_tail = coords1;
    }
    if ((rc = launch_conv_dbg(p, s))) return rc;
  }
  // ---- GRU (model_utils.py:138-169) ----
  const int passes = v.small ? 1 : 2;
  for (int pass = 0; pass < passes; ++pass) {
    int zr = pass == 0 ? P_ZR1 : P_ZR2, q = pass == 0 ? P_Q1 : P_Q2;
    ConvParams p = base_params(v, L, blob, zr, W.hx, v.hx, 0, B, h, w);
    hoist_inp(v, W, pass * 2 + 0, p);
    static const int stash = getenv("RAFT_B200_NO_STASH") ? 0 : 1;  // A/B knob (common.cuh: Stash)
    p.epi = EPI_ZR; p.f0 = W.Z; p.f1 = W.H; p.stash = stash;
    p.d0_hi = W.qx.hi; p.d0_lo = W.qx.lo; p.d0_stride = v.hx; p.d0_choff = 0;
    if ((rc = launch_conv_dbg(p, s))) return rc;
    p = base_params(v, L, blob, q, W.qx, v.hx, 0, B, h, w);
    hoist_inp(v, W, pass * 2 + 1, p);
    p.epi = EPI_Q; p.f0 = W.Z; p.f1 = W.H; p.stash = stash;
    p.d0_hi = W.hx.hi; p.d0_lo = W.hx.lo; p.d0_stride = v.hx; p.d0_choff = 0;
    if ((rc = launch_conv_dbg(p, s))) return rc;
  }
  // ---- flow head (model_utils.py:131-135) + coords1 += delta (RAFT.py:102) ----
  // conv2 (3x3, fh -> 2) runs as an N = 16 implicit GEMM on 55 CTAs (~15 us at batch 1).  Folding it into conv1's epilogue
  // (18 per-pixel dot products per 16-channel group + a gather kernel, no FH store) was built in round 2: parity-green and
  // 2.2 % SLOWER per iteration at batch 1, 5 % at batch 8 (same-box ABAB, profiles/r02_notes.md) -- removed again.
  {
    ConvParams p = base_params(v, L, blob, P_FH1, W.hx, v.hx, 0, B, h, w);
    set_act(p, ACT_RELU, W.fh, v.fh, 0);
    if ((rc = launch_conv_dbg(p, s))) return rc;
    p = base_params(v, L, blob, P_FH2, W.fh, v.fh, 0, B, h, w);
    p.epi = EPI_DELTA; p.f1 = coords1; p.f2 = delta_out;
    // 36 k-iterations on 55 CTAs at batch 1 while 93 SMs idle: two CTAs per pixel tile, half of the channel chunks each
    // (conv_tc.cu, split-K over a cluster when the tiles fit one wave of CTA pairs; the same two-halves sum on one CTA
    // otherwise, so batched and per-sample runs stay bit-identical).  RAFT_B200_NO_SPLITK=1: one accumulator.
    static const bool no_splitk = getenv("RAFT_B200_NO_SPLITK") != nullptr;
    p.split_k = no_splitk ? 0 : 1;
    if ((rc = launch_conv_dbg(p, s))) return rc;
  }
  // ---- mask head (model_utils.py:180-183); only the last iteration's mask is ever consumed ----
  if (mask_out) {
    RB_REQUIRE(!v.small, RB_ERR_UNSUPPORTED, "raft-small has no mask head (model_utils.py:194)");
    ConvParams p = base_params(v, L, blob, P_MASK0, W.hx, v.hx, 0, B, h, w);
    set_act(p, ACT_RELU, W.fh, v.fh, 0);
    if ((rc = launch_conv_dbg(p, s))) return rc;
    p = base_params(v, L, blob, P_MASK2, W.fh, v.fh, 0, B, h, w);
    p.epi = EPI_F32; p.f0 = mask_out; p.scale = 0.25f;
    if ((rc = launch_conv_dbg(p, s))) return rc;
  }
  return RB_OK;
}

// conv over the `inp` channels only (+bias) of the four GRU convs -> W.pre[0..3] (fp32)
static int precompute_inp(const Variant& v, const void* blob, void* wsp, int B, int h, int w, cudaStream_t s) {
  if (!can_hoist(v)) return RB_OK;
  const size_t npix = (size_t)B * h * w;
  const PackedLayout L = packed_layout(v);
  const Workspace W = workspace_layout(v, npix, wsp);
  const int ids[4] = {P_ZR1, P_Q1, P_ZR2, P_Q2};
  for (int i = 0; i < 4; ++i) {
    ConvParams p = base_params(v, L, blob, ids[i], W.hx, v.hx, 0, B, h, w);  // inp lives in HX and QX alike
    p.ck_begin = v.hidden / 64; p.ck_count = v.ctx / 64; p.ck_skip_at = 1 << 20; p.ck_skip = 0;
    p.epi = EPI_F32; p.f0 = W.pre[i]; p.scale = 1.f;
    int rc = launch_conv(p, s);
    if (rc) return rc;
  }
  return RB_OK;
}

}  // namespace rb

using namespace rb;

static int check_shape(const char* fn, int B, int h, int w) {
  RB_REQUIRE(B > 0 && h > 0 && w > 0 && (size_t)B * h * w < (1u << 30), RB_ERR_BAD_SHAPE, "%s: bad shape B=%d h=%d w=%d",
             fn, B, h, w);
  return RB_OK;
}

extern "C" int rb_debug_set_buffer(void* buf) {
  g_dbg = reinterpret_cast<long long*>(buf);
  return RB_OK;
}

extern "C" int rb_update_num_convs(int small) { return variant(small).nref; }

extern "C" const char* rb_update_conv_name(int small, int i) {
  const Variant& v = variant(small);
  if (i < 0 || i >= v.nref) return nullptr;
  return v.ref[i].name;
}

extern "C" int rb_update_conv_shape(int small, int i, int* kh, int* kw, int* cin, int* cout) {
  const Variant& v = variant(small);
  RB_REQUIRE(i >= 0 && i < v.nref, RB_ERR_BAD_ARG, "rb_update_conv_shape: index %d out of range", i);
  if (kh) *kh = v.ref[i].kh;
  if (kw) *kw = v.ref[i].kw;
  if (cin) *cin = v.ref[i].cin;
  if (cout) *cout = v.ref[i].cout;
  return RB_OK;
}

extern "C" int rb_update_weights_bytes(int small, size_t* bytes) {
  RB_REQUIRE(bytes, RB_ERR_BAD_ARG, "rb_update_weights_bytes: null output");
  *bytes = packed_layout(variant(small)).total;
  return RB_OK;
}

// Layout of packed conv `id` (0 .. 11 in the order convc1, convc2, convf2, motion encoder conv, convz|r 1, convq1, convz|r 2,
// convq2, flow-head conv1, conv2, mask conv0, conv2; 100 = the tensor-core form of convf1, [cout_pad][7][64]) inside the blob.
// cout == 0: the variant does not have this conv.
extern "C" int rb_update_packed_conv(int small, int id, size_t* hi_off, size_t* lo_off, size_t* bias_off, int* kh, int* kw,
                                     int* cin_pad, int* cout, int* cout_pad) {
  const Variant& v = variant(small);
  const PackedLayout L = packed_layout(v);
  RB_REQUIRE((id >= 0 && id < P_COUNT) || id == 100, RB_ERR_BAD_ARG, "rb_update_packed_conv: id %d", id);
  const bool f1 = id == 100;
  if (hi_off) *hi_off = f1 ? L.f1t_hi : L.hi[id];
  if (lo_off) *lo_off = f1 ? L.f1t_lo : L.lo[id];
  if (bias_off) *bias_off = f1 ? L.f1t_bias : L.bias[id];
  if (kh) *kh = f1 ? 7 : L.kh[id];
  if (kw) *kw = f1 ? 1 : L.kw[id];
  if (cin_pad) *cin_pad = f1 ? 64 : v.pk[id].cin_pad;
  if (cout) *cout = f1 ? L.f1t_cout : L.cout[id];
  if (cout_pad) *cout_pad = f1 ? L.f1t_cout_pad : L.cout_pad[id];
  return RB_OK;
}

// Host-only: the blob rb_update_weights_pack uploads, written to host memory (no GPU needed; tests/test_packing.py).
extern "C" int rb_update_weights_pack_host(int small, const float* const* W_host, const float* const* b_host, void* host_blob,
                                           size_t blob_bytes) {
  const Variant& v = variant(small);
  const PackedLayout L = packed_layout(v);
  RB_REQUIRE(W_host && b_host && host_blob, RB_ERR_BAD_ARG, "rb_update_weights_pack: null pointer");
  RB_REQUIRE(blob_bytes >= L.total, RB_ERR_WORKSPACE, "rb_update_weights_pack: blob has %zu bytes, need %zu",
             blob_bytes, L.total);
  for (int i = 0; i < v.nref; ++i)
    RB_REQUIRE(W_host[i] && b_host[i], RB_ERR_BAD_ARG, "rb_update_weights_pack: missing weights for %s", v.ref[i].name);
  struct HostBlob {
    char* p;
    char* data() { return p; }
  } host{reinterpret_cast<char*>(host_blob)};
  memset(host_blob, 0, L.total);
  for (int id = 0; id < P_COUNT; ++id) {
    const PackedConv& pc = v.pk[id];
    if (pc.src0 < 0) continue;
    __half* hi = reinterpret_cast<__half*>(host.data() + L.hi[id]);
    __half* lo = reinterpret_cast<__half*>(host.data() + L.lo[id]);
    float* bias = reinterpret_cast<float*>(host.data() + L.bias[id]);
    const int taps = L.kh[id] * L.kw[id];
    int co_base = 0;
    for (int sidx = 0; sidx < 2; ++sidx) {
      int src = sidx == 0 ? pc.src0 : pc.src1;
      if (src < 0) continue;
      const RefConv& r = v.ref[src];
      RB_REQUIRE(r.cin <= pc.cin_pad, RB_ERR_BAD_SHAPE, "internal: cin_pad too small for %s", r.name);
      const float* Wsrc = W_host[src];  // HWIO
      for (int t = 0; t < taps; ++t)
        for (int ci = 0; ci < r.cin; ++ci)
          for (int co = 0; co < r.cout; ++co) {
            float val = Wsrc[((size_t)t * r.cin + ci) * r.cout + co];
            size_t o = ((size_t)(co_base + co) * taps + t) * pc.cin_pad + ci;
            split_f32(val, hi[o], lo[o]);
          }
      for (int co = 0; co < r.cout; ++co) bias[co_base + co] = b_host[src][co];
      co_base += r.cout;
    }
  }
  {
    const RefConv& f = v.ref[v.convf1_ref];
    memcpy(host.data() + L.f1_w, W_host[v.convf1_ref], (size_t)f.kh * f.kw * f.cin * f.cout * sizeof(float));
    memcpy(host.data() + L.f1_b, b_host[v.convf1_ref], (size_t)f.cout * sizeof(float));
    // tensor-core form: tap (ky, kx), flow channel c -> [co][ky][kx * 8 + c] (window pixel kx of 8, 8 channels per pixel)
    RB_REQUIRE(f.kh == 7 && f.kw == 7 && f.cin == 2, RB_ERR_BAD_SHAPE, "internal: convf1 is expected to be 7x7x2");
    __half* hi = reinterpret_cast<__half*>(host.data() + L.f1t_hi);
    __half* lo = reinterpret_cast<__half*>(host.data() + L.f1t_lo);
    float* bias = reinterpret_cast<float*>(host.data() + L.f1t_bias);
    const float* Wsrc = W_host[v.convf1_ref];
    for (int ky = 0; ky < 7; ++ky)
      for (int kx = 0; kx < 7; ++kx)
        for (int c = 0; c < 2; ++c)
          for (int co = 0; co < f.cout; ++co) {
            const size_t o = ((size_t)co * 7 + ky) * 64 + kx * 8 + c;
            split_f32(Wsrc[((size_t)(ky * 7 + kx) * 2 + c) * f.cout + co], hi[o], lo[o]);
          }
    for (int co = 0; co < f.cout; ++co) bias[co] = b_host[v.convf1_ref][co];
  }
  return RB_OK;
}

extern "C" int rb_update_weights_pack(int small, const float* const* W_host, const float* const* b_host,
                                      void* blob, size_t blob_bytes, void* stream) {
  RB_REQUIRE(blob, RB_ERR_BAD_ARG, "rb_update_weights_pack: null pointer");
  const size_t total = packed_layout(variant(small)).total;
  RB_REQUIRE(blob_bytes >= total, RB_ERR_WORKSPACE, "rb_update_weights_pack: blob has %zu bytes, need %zu", blob_bytes, total);
  std::vector<char> host(total, 0);
  int rc = rb_update_weights_pack_host(small, W_host, b_host, host.data(), total);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  RB_CHECK_CUDA(cudaMemcpyAsync(blob, host.data(), total, cudaMemcpyHostToDevice, s));
  RB_CHECK_CUDA(cudaStreamSynchronize(s));  // `host` dies at return; packing is an init-time call
  return RB_OK;
}

extern "C" int rb_update_workspace_bytes(int small, int B, int h, int w, size_t* bytes) {
  RB_REQUIRE(bytes, RB_ERR_BAD_ARG, "rb_update_workspace_bytes: null output");
  int rc = check_shape("rb_update_workspace_bytes", B, h, w);
  if (rc) return rc;
  *bytes = workspace_layout(variant(small), (size_t)B * h * w, nullptr).total;
  return RB_OK;
}

extern "C" int rb_update_set_state(int small, const void* weights, void* workspace, const float* net, const float* inp,
                                   int B, int h, int w, void* stream) {
  RB_REQUIRE(weights && workspace && net && inp, RB_ERR_BAD_ARG, "rb_update_set_state: null pointer");
  int rc = check_shape("rb_update_set_state", B, h, w);
  if (rc) return rc;
  const Variant& v = variant(small);
  size_t npix = (size_t)B * h * w;
  Workspace W = workspace_layout(v, npix, workspace);
  size_t n = npix * (v.hidden + v.ctx);
  set_state_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(net, inp, W, (int)npix, v.hidden,
                                                                                  v.ctx, v.hx);
  RB_CHECK_LAUNCH("set_state_kernel");
  return precompute_inp(v, weights, workspace, B, h, w, (cudaStream_t)stream);
}

extern "C" int rb_update_set_state_cnet(int small, const void* weights, void* workspace, const float* cnet, int B, int h,
                                        int w, void* stream) {
  RB_REQUIRE(weights && workspace && cnet, RB_ERR_BAD_ARG, "rb_update_set_state_cnet: null pointer");
  int rc = check_shape("rb_update_set_state_cnet", B, h, w);
  if (rc) return rc;
  const Variant& v = variant(small);
  size_t npix = (size_t)B * h * w;
  Workspace W = workspace_layout(v, npix, workspace);
  size_t n = npix * (v.hidden + v.ctx);
  set_state_cnet_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(cnet, W, (int)npix, v.hidden, v.ctx, v.hx);
  RB_CHECK_LAUNCH("set_state_cnet_kernel");
  return precompute_inp(v, weights, workspace, B, h, w, (cudaStream_t)stream);
}

extern "C" int rb_update_get_net(int small, const void* workspace, float* net, int B, int h, int w, void* stream) {
  RB_REQUIRE(workspace && net, RB_ERR_BAD_ARG, "rb_update_get_net: null pointer");
  int rc = check_shape("rb_update_get_net", B, h, w);
  if (rc) return rc;
  const Variant& v = variant(small);
  size_t npix = (size_t)B * h * w;
  Workspace W = workspace_layout(v, npix, const_cast<void*>(workspace));
  size_t n = npix * v.hidden;
  copy_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(W.H, net, n);
  RB_CHECK_LAUNCH("copy_f32_kernel");
  return RB_OK;
}

extern "C" int rb_update_lookup(int small, void* workspace, const float* pyramid, const float* coords1, int B,
                                int h, int w, void* stream) {
  RB_REQUIRE(workspace && pyramid && coords1, RB_ERR_BAD_ARG, "rb_update_lookup: null pointer");
  int rc = check_shape("rb_update_lookup", B, h, w);
  if (rc) return rc;
  const Variant& v = variant(small);
  Workspace W = workspace_layout(v, (size_t)B * h * w, workspace);
  return launch_lookup(pyramid, coords1, nullptr, W.corr.hi, W.corr.lo, v.corr_pad, B, h, w, v.radius,
                       (cudaStream_t)stream);
}

/* volume-free form of rb_update_lookup (F2): correlation features straight from the feature maps */
extern "C" int rb_update_lookup_otf(int small, void* workspace, const float* fmap1, const float* fmap2, const void* otf_workspace,
                                    const float* coords1, int B, int h, int w, int C, void* stream) {
  RB_REQUIRE(workspace && fmap1 && fmap2 && otf_workspace && coords1, RB_ERR_BAD_ARG, "rb_update_lookup_otf: null pointer");
  int rc = check_shape("rb_update_lookup_otf", B, h, w);
  if (rc) return rc;
  const Variant& v = variant(small);
  Workspace W = workspace_layout(v, (size_t)B * h * w, workspace);
  return launch_lookup_otf(fmap1, fmap2, reinterpret_cast<const float*>(otf_workspace), coords1, nullptr, W.corr.hi, W.corr.lo,
                           v.corr_pad, B, h, w, C, v.radius, (cudaStream_t)stream);
}

extern "C" int rb_update_set_corr(int small, void* workspace, const float* corr, int B, int h, int w,
                                  void* stream) {
  RB_REQUIRE(workspace && corr, RB_ERR_BAD_ARG, "rb_update_set_corr: null pointer");
  int rc = check_shape("rb_update_set_corr", B, h, w);
  if (rc) return rc;
  const Variant& v = variant(small);
  size_t npix = (size_t)B * h * w;
  Workspace W = workspace_layout(v, npix, workspace);
  size_t n = npix * v.corr_ch;
  set_corr_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(corr, W.corr, (int)npix, v.corr_ch,
                                                                                 v.corr_pad);
  RB_CHECK_LAUNCH("set_corr_kernel");
  return RB_OK;
}

extern "C" int rb_update_step(int small, const void* weights, void* workspace, float* coords1, float* delta_out,
                              float* mask_out, int B, int h, int w, void* stream) {
  RB_REQUIRE(weights && workspace && coords1, RB_ERR_BAD_ARG, "rb_update_step: null pointer");
  int rc = check_shape("rb_update_step", B, h, w);
  if (rc) return rc;
  return update_step(variant(small), weights, workspace, coords1, delta_out, mask_out, B, h, w, (cudaStream_t)stream);
}

extern "C" int rb_raft_iterate(int small, const void* weights, void* workspace, const float* pyramid,
                               float* coords1, float* mask_out, int B, int h, int w, int iters, void* stream) {
  RB_REQUIRE(weights && workspace && pyramid && coords1, RB_ERR_BAD_ARG, "rb_raft_iterate: null pointer");
  RB_REQUIRE(iters >= 1, RB_ERR_BAD_ARG, "rb_raft_iterate: iters=%d", iters);
  RB_REQUIRE(small || mask_out, RB_ERR_BAD_ARG, "rb_raft_iterate: raft-things needs mask_out");
  int rc = check_shape("rb_raft_iterate", B, h, w);
  if (rc) return rc;
  const Variant& v = variant(small);
  for (int it = 0; it < iters; ++it) {
    float* m = (it == iters - 1 && !small) ? mask_out : nullptr;
    if ((rc = update_step(v, weights, workspace, coords1, nullptr, m, B, h, w, (cudaStream_t)stream, pyramid))) return rc;
  }
  return RB_OK;
}
