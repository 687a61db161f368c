// F5 (output edge): forward-backward consistency (occlusion) check of a bidirectional flow pair.
// The test of Sundaram et al. 2010 / UnFlow (Meister et al. 2018): a pixel p whose displacement u = scale*f(p) is not
// undone by the other direction's flow at p + u, |u + g(p + u)|^2 >= alpha1 (|u|^2 + |g(p + u)|^2) + alpha2, is marked
// occluded.  g(p + u) is sampled bilinearly with corners x0 = floor(tx), x1 = min(x0 + 1, W - 1) (same for y); inside
// [0, W-1] x [0, H-1] that is the value the reference's truncating sampler (networks/utils.py:40-99) gives in real
// arithmetic.  A gather of a few MB per pair: HBM / L2 bound.
#include "common.cuh"

namespace rb {

constexpr int kConsistencyPx = 4;  // consecutive pixels per thread: one 32-bit store of the mask

__device__ __forceinline__ uint32_t consistency_code(const float2* __restrict__ g, float2 f, int x, int y, int H, int W,
                                                     float scale, float alpha1, float alpha2) {
  const float ux = scale * f.x, uy = scale * f.y;
  const float tx = (float)x + ux, ty = (float)y + uy;
  // written so that NaN displacements also count as leaving the frame
  if (!(tx >= 0.f && tx <= (float)(W - 1) && ty >= 0.f && ty <= (float)(H - 1))) return 2u;
  const float fx = floorf(tx), fy = floorf(ty);
  const int x0 = (int)fx, y0 = (int)fy;
  const int x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
  const float ax = tx - fx, ay = ty - fy;
  const float2 g00 = g[(size_t)y0 * W + x0], g01 = g[(size_t)y0 * W + x1];
  const float2 g10 = g[(size_t)y1 * W + x0], g11 = g[(size_t)y1 * W + x1];
  const float w00 = (1.f - ax) * (1.f - ay), w01 = ax * (1.f - ay), w10 = (1.f - ax) * ay, w11 = ax * ay;
  const float gx = scale * (w00 * g00.x + w01 * g01.x + w10 * g10.x + w11 * g11.x);
  const float gy = scale * (w00 * g00.y + w01 * g01.y + w10 * g10.y + w11 * g11.y);
  const float sx = ux + gx, sy = uy + gy;
  const float lhs = sx * sx + sy * sy;
  const float rhs = alpha1 * (ux * ux + uy * uy + gx * gx + gy * gy) + alpha2;
  return lhs >= rhs ? 1u : 0u;
}

// grid.y = direction (0: fw against bw -> occ_fw, 1: bw against fw -> occ_bw); one thread per kConsistencyPx
// consecutive pixels of one row.
__global__ void flow_consistency_kernel(const float2* __restrict__ flow_fw, const float2* __restrict__ flow_bw,
                                        uint8_t* __restrict__ occ_fw, uint8_t* __restrict__ occ_bw, int B, int H, int W,
                                        float scale, float alpha1, float alpha2) {
  const int nq = (W + kConsistencyPx - 1) / kConsistencyPx;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * H * nq) return;
  const bool bw = blockIdx.y != 0;
  const float2* f = bw ? flow_bw : flow_fw;
  const float2* g = bw ? flow_fw : flow_bw;
  uint8_t* occ = bw ? occ_bw : occ_fw;
  const size_t row = i / nq;  // b * H + y
  const int y = (int)(row % H), xs = (int)(i % nq) * kConsistencyPx;
  const size_t b = row / H, o = row * W + xs;
  g += b * H * W;
  const int n = min(kConsistencyPx, W - xs);
  uint32_t codes = 0;
#pragma unroll
  for (int k = 0; k < kConsistencyPx; ++k)
    if (k < n) codes |= consistency_code(g, f[o + k], xs + k, y, H, W, scale, alpha1, alpha2) << (8 * k);
  if (n == kConsistencyPx && ((uintptr_t)(occ + o) & 3) == 0) {
    *reinterpret_cast<uint32_t*>(occ + o) = codes;
  } else {
    for (int k = 0; k < n; ++k) occ[o + k] = (uint8_t)(codes >> (8 * k));
  }
}

}  // namespace rb

using namespace rb;

extern "C" int rb_flow_consistency(const float* flow_fw, const float* flow_bw, uint8_t* occ_fw, uint8_t* occ_bw, int B,
                                   int H, int W, float scale, float alpha1, float alpha2, void* stream) {
  RB_REQUIRE(flow_fw && flow_bw && occ_fw && occ_bw, RB_ERR_BAD_ARG, "rb_flow_consistency: null pointer");
  RB_REQUIRE(((uintptr_t)flow_fw & 7) == 0 && ((uintptr_t)flow_bw & 7) == 0, RB_ERR_BAD_ARG,
             "rb_flow_consistency: flows must be 8-byte aligned (float2 loads)");
  RB_REQUIRE(B > 0 && H > 0 && W > 0, RB_ERR_BAD_SHAPE, "rb_flow_consistency: bad shape B=%d H=%d W=%d", B, H, W);
  RB_REQUIRE(isfinite(scale) && scale > 0.f, RB_ERR_BAD_ARG, "rb_flow_consistency: scale must be > 0, got %g",
             (double)scale);
  RB_REQUIRE(isfinite(alpha1) && isfinite(alpha2) && alpha1 >= 0.f && alpha2 >= 0.f, RB_ERR_BAD_ARG,
             "rb_flow_consistency: alpha1, alpha2 must be finite and >= 0, got %g, %g", (double)alpha1, (double)alpha2);
  const size_t n = (size_t)B * H * ((W + kConsistencyPx - 1) / kConsistencyPx);
  RB_REQUIRE((n + 255) / 256 <= 0x7fffffffu, RB_ERR_BAD_SHAPE, "rb_flow_consistency: B*H*W too large");
  const dim3 grid((unsigned)((n + 255) / 256), 2);
  flow_consistency_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float2*>(flow_fw), reinterpret_cast<const float2*>(flow_bw), occ_fw, occ_bw, B, H, W, scale,
      alpha1, alpha2);
  RB_CHECK_LAUNCH("flow_consistency_kernel");
  return RB_OK;
}
