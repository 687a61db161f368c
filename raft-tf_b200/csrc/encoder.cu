// F1 (SURVEY 8f): feature / context encoders on the same tensor-core conv kernels as the update block.
// Reference: networks/model_utils.py:6-105 (norm_func, ResidualBlock, BottleneckBlock, BasicEncoder,
// SmallEncoder) and networks/RAFT.py:53-76 (2x-1 preprocessing, fnet = instance norm, cnet = batch norm
// (things) / none (small)).
//
// Activations are split fp16 tensors [pixel][Cpad] (Cpad = channels rounded up to 64, pad = 0).
//   stride-1 convs  -> conv_tc implicit GEMM directly on the activation (TMA zero fill = TF SAME);
//   strided convs   -> (3x3 s2, 1x1 s2) the same kernel over a strided input VIEW (ConvParams, common.cuh): TMA element
//                      strides deliver every second pixel of the box, TF's asymmetric SAME offsets
//                      (pad_before = total/2) are the tile's start coordinates -- no gather pass;
//   7x7 s2 stem     -> one pass writes the 2x-1 image as a zero-padded space-to-depth tensor (2x2 pixels x 3 channels =
//                      12 of 16 channels per cell); a 7x7 stride-2 window is 4x4 such cells, and the 4 cells of one
//                      window row are 64 CONTIGUOUS channels, so the stem is a 4x1 conv (K = 4 x 64) over a view whose
//                      pixels overlap (x pitch 16 channels, extent 64) -- 7 MB instead of the 86 MB im2col of round 1;
//   instance norm   -> conv writes raw fp32, a two-stage deterministic reduction gives per-(sample,
//                      channel) mean / biased variance, one pass applies (x-mean)*rstd (+ReLU, + the
//                      residual add and final ReLU of the block) and re-splits;
//   batch norm      -> folded into the conv weights/bias at pack time (inference statistics);
//   none            -> bias + ReLU in the conv epilogue.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"

namespace rb {

static inline size_t al(size_t v, size_t a = 1024) { return (v + a - 1) / a * a; }
static inline int pad64(int c) { return (c + 63) / 64 * 64; }

enum { NORM_NONE = 0, NORM_INSTANCE = 1, NORM_BATCH = 2 };

struct EncConv {
  const char* name;  // relative to the encoder scope, e.g. "layer2/0/downsample.0"
  int k, stride, cin, cout;
  const char* norm;  // scope of the following norm ("" = none)
};

// order = execution order; names follow the reference's variable scopes
static const EncConv kBasicConvs[] = {
    {"conv1", 7, 2, 3, 64, "norm1"},
    {"layer1/0/conv1", 3, 1, 64, 64, "layer1/0/norm1"}, {"layer1/0/conv2", 3, 1, 64, 64, "layer1/0/norm2"},
    {"layer1/1/conv1", 3, 1, 64, 64, "layer1/1/norm1"}, {"layer1/1/conv2", 3, 1, 64, 64, "layer1/1/norm2"},
    {"layer2/0/conv1", 3, 2, 64, 96, "layer2/0/norm1"}, {"layer2/0/conv2", 3, 1, 96, 96, "layer2/0/norm2"},
    {"layer2/0/downsample.0", 1, 2, 64, 96, "layer2/0/downsample.1"},
    {"layer2/1/conv1", 3, 1, 96, 96, "layer2/1/norm1"}, {"layer2/1/conv2", 3, 1, 96, 96, "layer2/1/norm2"},
    {"layer3/0/conv1", 3, 2, 96, 128, "layer3/0/norm1"}, {"layer3/0/conv2", 3, 1, 128, 128, "layer3/0/norm2"},
    {"layer3/0/downsample.0", 1, 2, 96, 128, "layer3/0/downsample.1"},
    {"layer3/1/conv1", 3, 1, 128, 128, "layer3/1/norm1"}, {"layer3/1/conv2", 3, 1, 128, 128, "layer3/1/norm2"},
    {"conv2", 1, 1, 128, -1, ""}};
static const EncConv kSmallConvs[] = {
    {"conv1", 7, 2, 3, 32, "norm1"},
    {"layer1/0/conv1", 1, 1, 32, 8, "layer1/0/norm1"}, {"layer1/0/conv2", 3, 1, 8, 8, "layer1/0/norm2"},
    {"layer1/0/conv3", 1, 1, 8, 32, "layer1/0/norm3"},
    {"layer1/1/conv1", 1, 1, 32, 8, "layer1/1/norm1"}, {"layer1/1/conv2", 3, 1, 8, 8, "layer1/1/norm2"},
    {"layer1/1/conv3", 1, 1, 8, 32, "layer1/1/norm3"},
    {"layer2/0/conv1", 1, 1, 32, 16, "layer2/0/norm1"}, {"layer2/0/conv2", 3, 2, 16, 16, "layer2/0/norm2"},
    {"layer2/0/conv3", 1, 1, 16, 64, "layer2/0/norm3"}, {"layer2/0/downsample.0", 1, 2, 32, 64, "layer2/0/downsample.1"},
    {"layer2/1/conv1", 1, 1, 64, 16, "layer2/1/norm1"}, {"layer2/1/conv2", 3, 1, 16, 16, "layer2/1/norm2"},
    {"layer2/1/conv3", 1, 1, 16, 64, "layer2/1/norm3"},
    {"layer3/0/conv1", 1, 1, 64, 24, "layer3/0/norm1"}, {"layer3/0/conv2", 3, 2, 24, 24, "layer3/0/norm2"},
    {"layer3/0/conv3", 1, 1, 24, 96, "layer3/0/norm3"}, {"layer3/0/downsample.0", 1, 2, 64, 96, "layer3/0/downsample.1"},
    {"layer3/1/conv1", 1, 1, 96, 24, "layer3/1/norm1"}, {"layer3/1/conv2", 3, 1, 24, 24, "layer3/1/norm2"},
    {"layer3/1/conv3", 1, 1, 24, 96, "layer3/1/norm3"},
    {"conv2", 1, 1, 96, -1, ""}};

struct EncDesc {
  const EncConv* convs;
  int n;
};
static inline EncDesc enc_desc(int small) {
  return small ? EncDesc{kSmallConvs, (int)(sizeof(kSmallConvs) / sizeof(EncConv))}
               : EncDesc{kBasicConvs, (int)(sizeof(kBasicConvs) / sizeof(EncConv))};
}

// packed form of one conv: [cout_pad][kh*kw][cin_pad]; the stem as [cout_pad][4 cell rows][4 cells x 16]
struct EncPacked {
  int kh, kw, cin_pad, cout, cout_pad;
  size_t hi, lo, bias;
};
static void enc_packed_layout(int small, int out_dim, std::vector<EncPacked>& P, size_t* total) {
  EncDesc d = enc_desc(small);
  P.resize(d.n);
  size_t off = 0;
  for (int i = 0; i < d.n; ++i) {
    const EncConv& c = d.convs[i];
    EncPacked& p = P[i];
    const int cout = c.cout < 0 ? out_dim : c.cout;
    const bool stem = c.k == 7;  // 4x1 conv over the space-to-depth view
    p.kh = stem ? 4 : c.k;
    p.kw = stem ? 1 : c.k;
    p.cin_pad = stem ? 64 : pad64(c.cin);
    p.cout = cout;
    p.cout_pad = (cout + 15) / 16 * 16;
    size_t plane = (size_t)p.cout_pad * p.kh * p.kw * p.cin_pad * sizeof(__half);
    p.hi = off; off = al(off + plane, 256);
    p.lo = off; off = al(off + plane, 256);
    p.bias = off; off = al(off + (size_t)p.cout_pad * sizeof(float), 256);
  }
  *total = off;
}

// ---- kernels ----------------------------------------------------------------------------------------
// Stem input: the 2x-1 image (RAFT.py:53-59) as a zero-padded space-to-depth tensor.  Padded image row r' = r + pt
// (TF SAME: pt = total/2 rows of zeros before), cell (Y, X) holds rows 2Y, 2Y+1 and columns 2X, 2X+1: channel
// (dy*2 + dx)*3 + c of 16 (12..15 = 0).  Output pixel (oy, ox) of the 7x7 stride-2 conv reads cells (oy..oy+3, ox..ox+3).
// One thread per cell, each cell written once, [B][Hp][Wp][16] (the conv's view overlaps them).
__global__ void enc_stem_s2d_kernel(const float* __restrict__ img, __half* __restrict__ out_hi, __half* __restrict__ out_lo, int B,
                                    int H, int W, int pt, int pl, int Hp, int Wp) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * Hp * Wp) return;
  const int X = i % Wp, Y = (i / Wp) % Hp, b = i / ((size_t)Wp * Hp);
  __align__(16) __half hi[16], lo[16];
#pragma unroll
  for (int j = 12; j < 16; ++j) hi[j] = lo[j] = __float2half_rn(0.f);
  const float* base = img + (size_t)b * H * W * 3;
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const int r = 2 * Y + dy - pt, q = 2 * X + dx - pl;
      const bool in = r >= 0 && r < H && q >= 0 && q < W;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int j = (dy * 2 + dx) * 3 + c;
        if (in) split_f32(2.0f * __ldg(base + ((size_t)r * W + q) * 3 + c) - 1.0f, hi[j], lo[j]);
        else hi[j] = lo[j] = __float2half_rn(0.f);  // SAME zero padding is applied AFTER the 2x-1 preprocessing
      }
    }
  const uint4* h4 = reinterpret_cast<const uint4*>(hi);
  const uint4* l4 = reinterpret_cast<const uint4*>(lo);
  const size_t o = (((size_t)b * Hp + Y) * Wp + X) * 16;
  reinterpret_cast<uint4*>(out_hi + o)[0] = h4[0]; reinterpret_cast<uint4*>(out_hi + o)[1] = h4[1];
  reinterpret_cast<uint4*>(out_lo + o)[0] = l4[0]; reinterpret_cast<uint4*>(out_lo + o)[1] = l4[1];
}

// instance-norm statistics, stage 1: per (sample, pixel strip) partial sum / sum of squares per channel
__global__ void inorm_partial_kernel(const float* __restrict__ x, double* __restrict__ part, int npx, int C, int strips) {
  const int b = blockIdx.y, strip = blockIdx.x, c = threadIdx.x % C, lane_px = threadIdx.x / C;
  const int rows = blockDim.x / C;
  const int per = (npx + strips - 1) / strips;
  const int p0 = strip * per, p1 = min(p0 + per, npx);
  double s = 0.0, s2 = 0.0;
  for (int p = p0 + lane_px; p < p1; p += rows) {
    const float v = x[((size_t)b * npx + p) * C + c];
    s += v;
    s2 += (double)v * v;
  }
  extern __shared__ double sh[];
  sh[threadIdx.x] = s;
  sh[blockDim.x + threadIdx.x] = s2;
  __syncthreads();
  if (lane_px == 0) {
    for (int r = 1; r < rows; ++r) { s += sh[r * C + c]; s2 += sh[blockDim.x + r * C + c]; }
    part[(((size_t)b * strips + strip) * 2 + 0) * C + c] = s;
    part[(((size_t)b * strips + strip) * 2 + 1) * C + c] = s2;
  }
}
// stage 2: mean and 1/sqrt(var+eps) (biased variance, eps 1e-5: tensorpack InstanceNorm).
// One block per (sample, channel): the strips are summed by a fixed-shape tree (deterministic).
__global__ void inorm_final_kernel(const double* __restrict__ part, float2* __restrict__ stat, int npx, int C, int strips) {
  const int b = blockIdx.y, c = blockIdx.x, t = threadIdx.x;
  __shared__ double s1[256], s2[256];
  double a = 0.0, q = 0.0;
  for (int k = t; k < strips; k += 256) {
    a += part[(((size_t)b * strips + k) * 2 + 0) * C + c];
    q += part[(((size_t)b * strips + k) * 2 + 1) * C + c];
  }
  s1[t] = a; s2[t] = q;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) { s1[t] += s1[t + w]; s2[t] += s2[t + w]; }
    __syncthreads();
  }
  if (t == 0) {
    const double mean = s1[0] / npx;
    const double var = fmax(s2[0] / npx - mean * mean, 0.0);
    stat[b * C + c] = make_float2((float)mean, (float)(1.0 / sqrt(var + 1e-5)));
  }
}
// y = (x-mean)*rstd [ReLU]; optionally out = relu(res + y) (ResidualBlock :31-35); -> split [px][Cpad].
// 8 channels per thread (C is a multiple of 8 for every encoder layer).
__global__ void inorm_apply_kernel(const float* __restrict__ x, const float2* __restrict__ stat, const __half* __restrict__ res_hi,
                                   const __half* __restrict__ res_lo, int res_stride, __half* __restrict__ out_hi,
                                   __half* __restrict__ out_lo, int out_stride, int B, int npx, int C, int relu) {
  const int c8 = C / 8;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * npx * c8) return;
  const int c = (i % c8) * 8;
  const size_t px = i / c8;
  const int b = px / npx;
  const float4 x0 = *reinterpret_cast<const float4*>(x + px * C + c), x1 = *reinterpret_cast<const float4*>(x + px * C + c + 4);
  float v[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
  __align__(16) __half rh[8], rl[8];
  if (res_hi) {
    *reinterpret_cast<uint4*>(rh) = *reinterpret_cast<const uint4*>(res_hi + px * res_stride + c);
    *reinterpret_cast<uint4*>(rl) = *reinterpret_cast<const uint4*>(res_lo + px * res_stride + c);
  }
  __align__(16) __half oh[8], ol[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float2 st = stat[b * C + c + k];
    float y = (v[k] - st.x) * st.y;
    if (relu) y = fmaxf(y, 0.f);
    if (res_hi) y = fmaxf(join_f32(rh[k], rl[k]) + y, 0.f);
    split_f32(y, oh[k], ol[k]);
  }
  *reinterpret_cast<uint4*>(out_hi + px * out_stride + c) = *reinterpret_cast<const uint4*>(oh);
  *reinterpret_cast<uint4*>(out_lo + px * out_stride + c) = *reinterpret_cast<const uint4*>(ol);
}
// ---- workspace -----------------------------------------------------------------------------------------
struct EncWs {
  SplitPtr act[4];  // rotating activation buffers
  SplitPtr col;     // space-to-depth cells of the stem
  float* f32;       // raw conv output awaiting instance norm
  double* part;     // instance-norm partial sums [B][strips][2][C]
  size_t part_cap;  // strips * C it can hold per sample
  float2* stat;
  size_t total;
};
constexpr int kStrips = 256;

static EncWs enc_ws_layout(int small, int B, int H, int W, void* base) {
  EncWs w;
  char* b = reinterpret_cast<char*>(base);
  size_t off = 0;
  const size_t px2 = (size_t)B * ((H + 1) / 2) * ((W + 1) / 2);
  const int c0 = small ? 32 : 64;
  // the widest activation is at 1/2 resolution (pad64(c0) channels); 1/4 and 1/8 tensors are smaller
  const size_t act_plane = al(px2 * pad64(small ? 64 : 128) * sizeof(__half) / 1);  // generous: covers px4*128, px8*128
  for (int i = 0; i < 4; ++i) {
    w.act[i].hi = reinterpret_cast<__half*>(b + off); off += act_plane;
    w.act[i].lo = reinterpret_cast<__half*>(b + off); off += act_plane;
  }
  // stem input cells: (Ho+3) x (Wo+3) x 16; the overlapping view reads up to cell Wo+2 of a row
  const size_t col_plane = al((size_t)B * ((H + 1) / 2 + 3) * ((W + 1) / 2 + 3) * 16 * sizeof(__half));
  w.col.hi = reinterpret_cast<__half*>(b + off); off += col_plane;
  w.col.lo = reinterpret_cast<__half*>(b + off); off += col_plane;
  w.f32 = reinterpret_cast<float*>(b + off); off += al(px2 * (size_t)(small ? 64 : 128) * sizeof(float));
  // strips: kStrips for the stand-alone statistics pass, 4 per pixel tile when the conv epilogue produces them
  const size_t fused_cap = (size_t)4 * conv_tc_tiles_per_image((H + 1) / 2, (W + 1) / 2) * 128;
  w.part_cap = fused_cap > (size_t)kStrips * 256 ? fused_cap : (size_t)kStrips * 256;
  w.part = reinterpret_cast<double*>(b + off); off += al((size_t)B * w.part_cap * 2 * sizeof(double));
  w.stat = reinterpret_cast<float2*>(b + off); off += al((size_t)B * 256 * sizeof(float2));
  (void)c0;
  w.total = off;
  return w;
}

static inline void same_pad(int n, int k, int s, int* before, int* out) {
  const int o = (n + s - 1) / s;
  int total = (o - 1) * s + k - n;
  if (total < 0) total = 0;
  *before = total / 2;
  *out = o;
}

struct EncRun {
  int small, norm, B;
  const char* blob;
  const std::vector<EncPacked>* P;
  EncWs ws;
  cudaStream_t s;
};

// conv i on `in` ([B,h,w] split, stride in_stride) -> `dst` split (if norm/epilogue produces split) ; returns out dims
static int enc_conv(const EncRun& R, int i, const float* img, SplitPtr in, int in_stride, int h, int w, int relu,
                    SplitPtr res, int res_stride, SplitPtr dst, int dst_stride, float* f32_out, int* oh_, int* ow_) {
  const EncConv& c = enc_desc(R.small).convs[i];
  const EncPacked& pk = (*R.P)[i];
  int oh = h, ow = w;
  ConvParams p;
  memset(&p, 0, sizeof(p));
  p.in_hi = in.hi; p.in_lo = in.lo; p.in_stride = in_stride; p.in_choff = 0; p.cin_pad = pk.cin_pad;
  if (c.k == 7) {  // stem: 4x1 conv over the space-to-depth view of the image
    int pt, pl;
    same_pad(h, c.k, c.stride, &pt, &oh);
    same_pad(w, c.k, c.stride, &pl, &ow);
    const int Hp = oh + 3, Wp = ow + 3;
    const size_t cells = (size_t)R.B * Hp * Wp;
    enc_stem_s2d_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, R.s>>>(img, R.ws.col.hi, R.ws.col.lo, R.B, h, w, pt, pl, Hp, Wp);
    RB_CHECK_LAUNCH("enc_stem_s2d_kernel");
    p.in_hi = R.ws.col.hi; p.in_lo = R.ws.col.lo;
    p.in_stride = 16;
    p.in_cext = 64;
    p.in_w = ow; p.in_h = Hp;
    p.in_rowpitch = Wp * 16;
    p.pad_explicit = 1; p.pad_x = 0; p.pad_y = 0;
  } else if (c.stride != 1) {  // strided view of the activation, TF SAME offsets
    int pt, pl;
    same_pad(h, c.k, c.stride, &pt, &oh);
    same_pad(w, c.k, c.stride, &pl, &ow);
    p.in_w = w; p.in_h = h;
    p.sx = p.sy = c.stride;
    p.pad_explicit = 1; p.pad_x = pl; p.pad_y = pt;
  }
  p.w_hi = reinterpret_cast<const __half*>(R.blob + pk.hi);
  p.w_lo = reinterpret_cast<const __half*>(R.blob + pk.lo);
  p.bias = reinterpret_cast<const float*>(R.blob + pk.bias);
  p.cout = pk.cout; p.cout_pad = pk.cout_pad; p.kh = pk.kh; p.kw = pk.kw;
  p.B = R.B; p.h = oh; p.w = ow;
  p.scale = 1.f;
  const bool has_norm = c.norm[0] != 0;
  const bool inorm = has_norm && R.norm == NORM_INSTANCE;
  int rc;
  if (f32_out) {  // final 1x1 conv: plain fp32 output
    p.epi = EPI_F32; p.f0 = f32_out;
    if ((rc = launch_conv(p, R.s))) return rc;
  } else if (inorm) {
    p.epi = EPI_F32; p.f0 = R.ws.f32;
    const int npx = oh * ow, C = pk.cout;
    // statistics, stage 1: by the conv's own epilogue (per pixel tile and lane quarter) when it runs on the tensor-core
    // kernel with the 16-channel epilogue, else by a pass over the fp32 output
    int strips = kStrips;
    const int fused_strips = 4 * conv_tc_tiles_per_image(oh, ow);
    if (conv_tc_fused_stats_ok(p) && (size_t)fused_strips * C <= R.ws.part_cap) {
      p.stat_part = R.ws.part;
      p.stat_strips = strips = fused_strips;
    }
    if ((rc = launch_conv(p, R.s))) return rc;
    if (!p.stat_part) {
      const int rows = max(1, 256 / C);
      dim3 g1(kStrips, R.B);
      inorm_partial_kernel<<<g1, rows * C, 2 * rows * C * sizeof(double), R.s>>>(R.ws.f32, R.ws.part, npx, C, kStrips);
      RB_CHECK_LAUNCH("inorm_partial_kernel");
    }
    inorm_final_kernel<<<dim3(C, R.B), 256, 0, R.s>>>(R.ws.part, R.ws.stat, npx, C, strips);
    RB_CHECK_LAUNCH("inorm_final_kernel");
    size_t n = (size_t)R.B * npx * (C / 8);
    inorm_apply_kernel<<<(unsigned)((n + 255) / 256), 256, 0, R.s>>>(R.ws.f32, R.ws.stat, res.hi, res.lo, res_stride, dst.hi,
                                                                     dst.lo, dst_stride, R.B, npx, C, relu);
    RB_CHECK_LAUNCH("inorm_apply_kernel");
  } else {  // batch norm folded into W/b, or no norm: bias (+ReLU) in the epilogue
    p.epi = EPI_ACT; p.act = relu ? ACT_RELU : ACT_NONE;
    p.d0_hi = dst.hi; p.d0_lo = dst.lo; p.d0_stride = dst_stride; p.d0_choff = 0;
    p.res_hi = res.hi; p.res_lo = res.lo; p.res_stride = res_stride;  // block output relu(x + y) in the same epilogue
    if ((rc = launch_conv(p, R.s))) return rc;
  }
  *oh_ = oh;
  *ow_ = ow;
  return RB_OK;
}

static int enc_forward(const EncRun& R, const float* image, float* out, int H, int W, int out_dim) {
  const SplitPtr none{nullptr, nullptr};
  const SplitPtr* A = R.ws.act;
  int h, w, rc, ci = 0;
  const EncConv* C = enc_desc(R.small).convs;
  // stem: conv1 7x7 s2 + norm + relu  (model_utils.py:68-70 / 92-94)
  int c_cur = C[0].cout;
  if ((rc = enc_conv(R, ci++, image, none, 0, H, W, 1, none, 0, A[0], pad64(c_cur), nullptr, &h, &w))) return rc;
  int cur = 0;  // index of the buffer holding the block input
  for (int layer = 0; layer < 3; ++layer) {
    for (int blk = 0; blk < 2; ++blk) {
      const int stride = (blk == 0 && layer > 0) ? 2 : 1;
      const int t1 = (cur + 1) & 3, t2 = (cur + 2) & 3, t3 = (cur + 3) & 3;
      const int cin = c_cur;
      int oh, ow;
      if (!R.small) {  // ResidualBlock (model_utils.py:19-35)
        const int cout = C[ci].cout;
        if ((rc = enc_conv(R, ci, nullptr, A[cur], pad64(cin), h, w, 1, none, 0, A[t1], pad64(cout), nullptr, &oh, &ow))) return rc;
        SplitPtr res = A[cur];
        int res_stride = pad64(cin);
        if (stride != 1) {  // downsample.0 + downsample.1 (no ReLU) on the block input
          int dh, dw;
          if ((rc = enc_conv(R, ci + 2, nullptr, A[cur], pad64(cin), h, w, 0, none, 0, A[t3], pad64(cout), nullptr, &dh, &dw))) return rc;
          res = A[t3];
          res_stride = pad64(cout);
        }
        if ((rc = enc_conv(R, ci + 1, nullptr, A[t1], pad64(cout), oh, ow, 1, res, res_stride, A[t2], pad64(cout), nullptr, &oh, &ow)))
          return rc;
        ci += (stride != 1) ? 3 : 2;
        cur = t2; c_cur = cout; h = oh; w = ow;
      } else {  // BottleneckBlock (model_utils.py:37-57)
        const int cmid = C[ci].cout, cout = C[ci + 2].cout;
        if ((rc = enc_conv(R, ci, nullptr, A[cur], pad64(cin), h, w, 1, none, 0, A[t1], pad64(cmid), nullptr, &oh, &ow))) return rc;
        if ((rc = enc_conv(R, ci + 1, nullptr, A[t1], pad64(cmid), h, w, 1, none, 0, A[t2], pad64(cmid), nullptr, &oh, &ow))) return rc;
        SplitPtr res = A[cur];
        int res_stride = pad64(cin);
        if (stride != 1) {
          int dh, dw;
          if ((rc = enc_conv(R, ci + 3, nullptr, A[cur], pad64(cin), h, w, 0, none, 0, A[t3], pad64(cout), nullptr, &dh, &dw))) return rc;
          res = A[t3];
          res_stride = pad64(cout);
        }
        // conv3 reads t2 and writes t1 (free again) with the residual fused
        if ((rc = enc_conv(R, ci + 2, nullptr, A[t2], pad64(cmid), oh, ow, 1, res, res_stride, A[t1], pad64(cout), nullptr, &oh, &ow)))
          return rc;
        ci += (stride != 1) ? 4 : 3;
        cur = t1; c_cur = cout; h = oh; w = ow;
      }
    }
  }
  // conv2: 1x1 to out_dim, no norm / activation (model_utils.py:76 / 100)
  int oh, ow;
  return enc_conv(R, ci, nullptr, A[cur], pad64(c_cur), h, w, 0, none, 0, none, 0, out, &oh, &ow);
}

}  // namespace rb

using namespace rb;

extern "C" int rb_encoder_num_convs(int small) { return enc_desc(small).n; }
extern "C" const char* rb_encoder_conv_name(int small, int i) {
  EncDesc d = enc_desc(small);
  return (i >= 0 && i < d.n) ? d.convs[i].name : nullptr;
}
extern "C" const char* rb_encoder_norm_name(int small, int i) {
  EncDesc d = enc_desc(small);
  return (i >= 0 && i < d.n) ? d.convs[i].norm : nullptr;
}
extern "C" int rb_encoder_conv_shape(int small, int i, int out_dim, int* k, int* stride, int* cin, int* cout) {
  EncDesc d = enc_desc(small);
  RB_REQUIRE(i >= 0 && i < d.n, RB_ERR_BAD_ARG, "rb_encoder_conv_shape: index %d out of range", i);
  if (k) *k = d.convs[i].k;
  if (stride) *stride = d.convs[i].stride;
  if (cin) *cin = d.convs[i].cin;
  if (cout) *cout = d.convs[i].cout < 0 ? out_dim : d.convs[i].cout;
  return RB_OK;
}
extern "C" int rb_encoder_weights_bytes(int small, int out_dim, size_t* bytes) {
  RB_REQUIRE(bytes && out_dim > 0, RB_ERR_BAD_ARG, "rb_encoder_weights_bytes: bad argument");
  std::vector<EncPacked> P;
  enc_packed_layout(small, out_dim, P, bytes);
  return RB_OK;
}

// Layout of conv i inside the packed blob (byte offsets of the hi / lo / bias planes and the packed geometry).
extern "C" int rb_encoder_packed_conv(int small, int out_dim, int i, size_t* hi_off, size_t* lo_off, size_t* bias_off, int* kh,
                                      int* kw, int* cin_pad, int* cout_pad) {
  std::vector<EncPacked> P;
  size_t total;
  enc_packed_layout(small, out_dim, P, &total);
  RB_REQUIRE(i >= 0 && i < (int)P.size() && out_dim > 0, RB_ERR_BAD_ARG, "rb_encoder_packed_conv: index %d out of range", i);
  if (hi_off) *hi_off = P[i].hi;
  if (lo_off) *lo_off = P[i].lo;
  if (bias_off) *bias_off = P[i].bias;
  if (kh) *kh = P[i].kh;
  if (kw) *kw = P[i].kw;
  if (cin_pad) *cin_pad = P[i].cin_pad;
  if (cout_pad) *cout_pad = P[i].cout_pad;
  return RB_OK;
}

// bn_host[i] (NORM_BATCH only): 4*cout floats [gamma | beta | mean/EMA | variance/EMA] of the norm after conv i.
// Host-only: the blob rb_encoder_weights_pack uploads, written to host memory (no GPU needed; tests/test_packing.py).
extern "C" int rb_encoder_weights_pack_host(int small, int norm, int out_dim, const float* const* W_host,
                                            const float* const* b_host, const float* const* bn_host, void* host_blob,
                                            size_t blob_bytes) {
  RB_REQUIRE(W_host && b_host && host_blob, RB_ERR_BAD_ARG, "rb_encoder_weights_pack: null pointer");
  RB_REQUIRE(norm >= 0 && norm <= 2, RB_ERR_BAD_ARG, "rb_encoder_weights_pack: norm %d", norm);
  std::vector<EncPacked> P;
  size_t total;
  enc_packed_layout(small, out_dim, P, &total);
  RB_REQUIRE(blob_bytes >= total, RB_ERR_WORKSPACE, "rb_encoder_weights_pack: blob has %zu bytes, need %zu", blob_bytes, total);
  EncDesc d = enc_desc(small);
  struct HostBlob {  // same interface as the std::vector<char> the loop below was written for
    char* p;
    char* data() { return p; }
  } host{reinterpret_cast<char*>(host_blob)};
  memset(host_blob, 0, total);
  for (int i = 0; i < d.n; ++i) {
    const EncConv& c = d.convs[i];
    const EncPacked& p = P[i];
    RB_REQUIRE(W_host[i] && b_host[i], RB_ERR_BAD_ARG, "rb_encoder_weights_pack: missing weights for %s", c.name);
    __half* hi = reinterpret_cast<__half*>(host.data() + p.hi);
    __half* lo = reinterpret_cast<__half*>(host.data() + p.lo);
    float* bias = reinterpret_cast<float*>(host.data() + p.bias);
    const int cout = p.cout, taps_ref = c.k * c.k;
    const bool stem = c.k == 7;
    const bool fold = norm == NORM_BATCH && c.norm[0] != 0;
    RB_REQUIRE(!fold || (bn_host && bn_host[i]), RB_ERR_BAD_ARG, "rb_encoder_weights_pack: missing BN statistics for %s", c.norm);
    for (int co = 0; co < cout; ++co) {
      double scale = 1.0, shift = 0.0;
      if (fold) {  // y = (conv + b - mean) / sqrt(var + eps) * gamma + beta
        const float* bn = bn_host[i];
        scale = (double)bn[co] / sqrt((double)bn[3 * cout + co] + 1e-5);
        shift = (double)bn[cout + co] - (double)bn[2 * cout + co] * scale;
      }
      for (int t = 0; t < taps_ref; ++t)
        for (int ci = 0; ci < c.cin; ++ci) {
          const float val = (float)(W_host[i][((size_t)t * c.cin + ci) * cout + co] * scale);
          size_t o = ((size_t)co * taps_ref + t) * p.cin_pad + ci;
          if (stem) {  // tap (ky, kx) = cell (ky/2, kx/2), sub-pixel (ky%2, kx%2): [co][cell row][cell x 16 + sub*3 + ci]
            const int ky = t / c.k, kx = t % c.k;
            o = ((size_t)co * 4 + ky / 2) * 64 + (kx / 2) * 16 + ((ky & 1) * 2 + (kx & 1)) * 3 + ci;
          }
          split_f32(val, hi[o], lo[o]);
        }
      bias[co] = (float)(b_host[i][co] * scale + shift);
    }
  }
  return RB_OK;
}

extern "C" int rb_encoder_weights_pack(int small, int norm, int out_dim, const float* const* W_host,
                                       const float* const* b_host, const float* const* bn_host, void* blob,
                                       size_t blob_bytes, void* stream) {
  RB_REQUIRE(blob, RB_ERR_BAD_ARG, "rb_encoder_weights_pack: null pointer");
  size_t total = 0;
  int rc = rb_encoder_weights_bytes(small, out_dim, &total);
  if (rc) return rc;
  RB_REQUIRE(blob_bytes >= total, RB_ERR_WORKSPACE, "rb_encoder_weights_pack: blob has %zu bytes, need %zu", blob_bytes, total);
  std::vector<char> host(total, 0);
  if ((rc = rb_encoder_weights_pack_host(small, norm, out_dim, W_host, b_host, bn_host, host.data(), total))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  RB_CHECK_CUDA(cudaMemcpyAsync(blob, host.data(), total, cudaMemcpyHostToDevice, s));
  RB_CHECK_CUDA(cudaStreamSynchronize(s));
  return RB_OK;
}

extern "C" int rb_encoder_workspace_bytes(int small, int B, int H, int W, size_t* bytes) {
  RB_REQUIRE(bytes && B > 0 && H >= 8 && W >= 8, RB_ERR_BAD_ARG, "rb_encoder_workspace_bytes: bad argument");
  *bytes = enc_ws_layout(small, B, H, W, nullptr).total;
  return RB_OK;
}

extern "C" int rb_encoder_forward(int small, int norm, const void* weights, const float* image, float* out, int B, int H,
                                  int W, int out_dim, void* workspace, size_t workspace_bytes, void* stream) {
  RB_REQUIRE(weights && image && out && workspace, RB_ERR_BAD_ARG, "rb_encoder_forward: null pointer");
  RB_REQUIRE(B > 0 && H >= 8 && W >= 8 && out_dim > 0 && out_dim <= 256, RB_ERR_BAD_SHAPE, "rb_encoder_forward: bad shape");
  RB_REQUIRE(norm >= 0 && norm <= 2, RB_ERR_BAD_ARG, "rb_encoder_forward: norm %d", norm);
  EncRun R;
  R.small = small; R.norm = norm; R.B = B;
  R.blob = reinterpret_cast<const char*>(weights);
  std::vector<EncPacked> P;
  size_t total;
  enc_packed_layout(small, out_dim, P, &total);
  R.P = &P;
  R.ws = enc_ws_layout(small, B, H, W, workspace);
  RB_REQUIRE(workspace_bytes >= R.ws.total, RB_ERR_WORKSPACE, "rb_encoder_forward: workspace has %zu bytes, need %zu",
             workspace_bytes, R.ws.total);
  R.s = (cudaStream_t)stream;
  return enc_forward(R, image, out, H, W, out_dim);
}
