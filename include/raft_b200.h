/*
 * raft_b200.h -- C ABI of the B200-native RAFT recurrent-inference hot path.
 *
 * The reference (gonglixue/RAFT-tf) has NO native/FFI boundary: its hot path is a set of Python
 * graph-building functions called from RAFT.network_graph (networks/RAFT.py:78-109).  Each entry
 * point below replaces one of those functions (cited per symbol); the Python mirrors in
 * raft-tf_b200/networks/ keep the reference's names and signatures and call these through ctypes.
 *
 * Conventions
 *  - every function returns an int status: 0 = RB_OK, negative = error (see enum); nothing throws
 *    or aborts; rb_last_error() returns a thread-local description of the last failure;
 *  - every data pointer is a DEVICE pointer to a caller-owned, contiguous buffer unless the
 *    parameter name ends in _host; tensors are NHWC fp32 exactly like the reference's TF tensors;
 *  - `stream` is a cudaStream_t passed as void*; calls only ENQUEUE work on it -- no hidden
 *    synchronisation, no hidden allocation (scratch comes from caller buffers sized by the
 *    *_bytes queries) -- so every call except rb_update_weights_pack is CUDA-graph capturable;
 *  - `small` selects raft-small (radius 3, hidden 96, context 64) vs raft-things (4, 128, 128),
 *    mirroring args.small (networks/RAFT.py:37-40).
 */
#ifndef RAFT_B200_H_
#define RAFT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  RB_OK = 0,
  RB_ERR_BAD_SHAPE = -1,
  RB_ERR_BAD_ARG = -2,
  RB_ERR_UNSUPPORTED = -3,
  RB_ERR_CUDA = -4,
  RB_ERR_WORKSPACE = -5
};

/* Arithmetic back end for the GEMM-shaped ops (corr build, update-block convs).
 *   RB_MATH_TC    tcgen05 tensor cores, fp16 hi/lo split operands, 3 MMAs per product,
 *                 fp32 accumulation in TMEM (error ~2^-22 relative per product);
 *   RB_MATH_SIMT  the same split operands multiplied on the fp32 CUDA cores (bring-up /
 *                 cross-check path; identical buffers and epilogues). */
enum { RB_MATH_TC = 0, RB_MATH_SIMT = 1 };

#define RB_NUM_LEVELS 4

int rb_version(void);
const char* rb_last_error(void);
/* Select the back end for subsequent calls on this thread (default RB_MATH_TC). */
int rb_set_math_mode(int mode);
int rb_get_math_mode(void);
/* Device selection.  The library carries its own CUDA runtime instance; its per-thread current device does not follow the
 * host framework's (torch.cuda.device(...), cudaSetDevice in another runtime).  Call this when the calling thread switches
 * GPUs, before the calls that enqueue work (their stream argument 0 = "default stream of the current device").
 * One process per GPU (torchrun) never needs it. */
int rb_set_device(int device);
/* Number of kernels this library has launched on the calling thread since the last reset. */
long long rb_launch_count(void);
void rb_launch_count_reset(void);

/* Profiling aid: when buf != NULL, rb_update_step records 8 globaltimer timestamps per CTA of each of its
 * tensor-core convs into buf (int64[n_convs][4096][8], launch order); NULL switches it off. */
int rb_debug_set_buffer(void* buf);

/* ---- A4: coords_grid(batch, ht, wd)  networks/utils.py:4-11 ----------------------------------
 * coords[b,y,x,0] = x, coords[b,y,x,1] = y. */
int rb_coords_grid(float* coords, int B, int h, int w, void* stream);

/* ---- A1: GetCorrPyramid(fmap1, fmap2, num_levels=4)  networks/model_utils.py:199-221 ----------
 * pyramid layout: level l (dims h_l = h >> l, w_l = w >> l, floor) is a dense fp32 array
 * [B*h*w, h_l, w_l]; levels are concatenated, level l starting at rb_corr_level_offset(). */
int rb_corr_pyramid_bytes(int B, int h, int w, size_t* bytes);
int rb_corr_level_offset(int B, int h, int w, int level, size_t* offset_floats, int* hl, int* wl);
int rb_corr_workspace_bytes(int B, int h, int w, int C, size_t* bytes);
int rb_corr_build(const float* fmap1, const float* fmap2, float* pyramid, int B, int h, int w,
                  int C, void* workspace, size_t workspace_bytes, void* stream);

/* ---- A2/A3: SampleCorr(corr_pyramid, coords, num_levels=4, radius)  model_utils.py:224-249 ----
 * with bilinear_sampler / tf_grid_sample semantics of networks/utils.py:39-103 (truncation toward
 * zero, index clamping, weights from the clamped x1/y1).  out: [B,h,w,4*(2r+1)^2] fp32, channel =
 * level*(2r+1)^2 + (x_off+r)*(2r+1) + (y_off+r). */
int rb_corr_lookup(const float* pyramid, const float* coords, float* out, int B, int h, int w,
                   int radius, void* stream);

/* ---- A3 (general form): bilinear_sampler(img, coords)  networks/utils.py:101-103 ---------------
 * img [n,H,W,1], coords [n,S,2] (x,y in pixels) -> out [n,S]; tf_grid_sample semantics (:39-99). */
int rb_bilinear_sample(const float* img, const float* coords, float* out, int n, int H, int W, int S,
                       void* stream);

/* ---- A14: tensorpack Conv2D(stride 1, padding 'same', use_bias) on fp32 NHWC tensors -----------
 * x [B,h,w,cin], W_host HWIO [kh,kw,cin,cout] and b_host [cout] (host pointers; b_host nullable),
 * y [B,h,w,cout] = act(conv(x,W)+b), act = ReLU if relu != 0.  Synchronises the stream once to upload
 * the packed kernel (stand-alone / test entry; the update block keeps its weights resident). */
int rb_conv2d_workspace_bytes(int B, int h, int w, int cin, int cout, int kh, int kw, size_t* bytes);
int rb_conv2d(const float* x, const float* W_host, const float* b_host, float* y, int B, int h, int w,
              int cin, int cout, int kh, int kw, int relu, void* workspace, size_t workspace_bytes,
              void* stream);
/* Same with tensorpack's `strides` argument (1 or 2; the encoders' stride-2 layers, model_utils.py:21,39,68,92):
 * y [B, ceil(h/stride), ceil(w/stride), cout], TensorFlow 'SAME' padding (pad before = total / 2, the odd one after).
 * The strided taps are read through TMA element strides -- no gathered copy of the input.  Same workspace query. */
int rb_conv2d_strided(const float* x, const float* W_host, const float* b_host, float* y, int B, int h, int w,
                      int cin, int cout, int kh, int kw, int stride, int relu, void* workspace,
                      size_t workspace_bytes, void* stream);

/* ---- A5-A11: BasicUpdateBlock / SmallUpdateBlock  model_utils.py:110-194 ----------------------
 * Weights: rb_update_num_convs(small) convolutions in the fixed order given by
 * rb_update_conv_name(small, i) (reference variable scopes, e.g. "update_block/gru/convz1");
 * W_host[i] is the HWIO fp32 kernel [kh,kw,cin,cout], b_host[i] the bias [cout] (host pointers,
 * as loaded from the reference's .npz).  The packed blob is device memory owned by the caller. */
int rb_update_num_convs(int small);
const char* rb_update_conv_name(int small, int i);
int rb_update_conv_shape(int small, int i, int* kh, int* kw, int* cin, int* cout);
int rb_update_weights_bytes(int small, size_t* bytes);
int rb_update_weights_pack(int small, const float* const* W_host, const float* const* b_host,
                           void* blob, size_t blob_bytes, void* stream);
/* Host-only forms (no GPU needed): the same blob written to host memory, and where packed conv `id` lives inside it
 * (id 0..11: convc1, convc2, convf2, motion-encoder conv, convz|r 1, convq1, convz|r 2, convq2, flow-head conv1, conv2, mask
 * conv0, conv2; 100: the tensor-core form of convf1).  Planes are [cout_pad][kh*kw][cin_pad] fp16 (hi, lo) + fp32 bias. */
int rb_update_weights_pack_host(int small, const float* const* W_host, const float* const* b_host, void* host_blob,
                                size_t blob_bytes);
int rb_update_packed_conv(int small, int id, size_t* hi_off, size_t* lo_off, size_t* bias_off, int* kh, int* kw,
                          int* cin_pad, int* cout, int* cout_pad);

/* Workspace holding the recurrent state (net), the context features (inp) and every per-iteration
 * activation.  Must be zero-filled by the caller once before first use (cudaMemset). */
int rb_update_workspace_bytes(int small, int B, int h, int w, size_t* bytes);
/* net = tanh(cnet[..., :hidden]) and inp = relu(cnet[..., hidden:]) (RAFT.py:85-87) are supplied
 * already activated: net [B,h,w,hidden], inp [B,h,w,context].  `weights` is the packed blob: the
 * iteration-invariant contribution of `inp` to the GRU convolutions is computed here, once per pair. */
int rb_update_set_state(int small, const void* weights, void* workspace, const float* net,
                        const float* inp, int B, int h, int w, void* stream);
/* Same from the raw context-encoder output cnet [B,h,w,hidden+context]: applies the split, tanh and relu of
 * RAFT.py:85-87 itself. */
int rb_update_set_state_cnet(int small, const void* weights, void* workspace, const float* cnet,
                             int B, int h, int w, void* stream);
int rb_update_get_net(int small, const void* workspace, float* net, int B, int h, int w,
                      void* stream);
/* Lookup written straight into the workspace in the layout the first conv consumes (fast path). */
int rb_update_lookup(int small, void* workspace, const float* pyramid, const float* coords1, int B,
                     int h, int w, void* stream);
/* Same slot filled from an fp32 [B,h,w,4*(2r+1)^2] tensor (functional BasicUpdateBlock mirror). */
int rb_update_set_corr(int small, void* workspace, const float* corr, int B, int h, int w,
                       void* stream);
/* One update-block application: flow = coords1 - coords_grid (RAFT.py:95), motion encoder, GRU,
 * flow head, coords1 += delta (RAFT.py:102).  delta_out (nullable) receives delta_flow [B,h,w,2];
 * mask_out (nullable) receives 0.25*mask [B,h,w,576] (things only; model_utils.py:180-183). */
int rb_update_step(int small, const void* weights, void* workspace, float* coords1,
                   float* delta_out, float* mask_out, int B, int h, int w, void* stream);
/* ---- A12: the loop of RAFT.network_graph (RAFT.py:91-102): iters x (lookup, update). ---------- */
int rb_raft_iterate(int small, const void* weights, void* workspace, const float* pyramid,
                    float* coords1, float* mask_out, int B, int h, int w, int iters, void* stream);

/* ---- F2 (SURVEY 8(f)): volume-free correlation -- GetCorrPyramid + SampleCorr (model_utils.py:199-249) without the
 * 4*N^2-byte volume.  Level l of the pyramid equals fmap1 . pool^l(fmap2)^T / sqrt(C) (pooling is linear), so each
 * iteration evaluates only the (2r+3) x (2r+3) entries per pixel and level that the bilinear taps can touch, as fp32
 * dot products against the pooled feature maps, and applies the same tap arithmetic as rb_corr_lookup.  Results equal
 * the materialised path up to the summation order / operand rounding of the dot products (parity is on the flow, 1e-3).
 * rb_corr_otf_prepare pools fmap2 once per pair into `workspace` (levels 1..3, fp32); C = 128 or 256. */
int rb_corr_otf_workspace_bytes(int B, int h, int w, int C, size_t* bytes);
int rb_corr_otf_prepare(const float* fmap2, void* workspace, size_t workspace_bytes, int B, int h, int w, int C,
                        void* stream);
int rb_corr_otf_lookup(const float* fmap1, const float* fmap2, const void* workspace, const float* coords,
                       float* out, int B, int h, int w, int C, int radius, void* stream);
/* lookup written straight into the update workspace (the volume-free counterpart of rb_update_lookup) */
int rb_update_lookup_otf(int small, void* workspace, const float* fmap1, const float* fmap2,
                         const void* otf_workspace, const float* coords1, int B, int h, int w, int C, void* stream);

/* ---- A13: RAFT.upsample_flow (RAFT.py:119-134) and upflow8 (utils.py:105-111) ----------------
 * flow = coords1 - coords_grid is formed inside; out: [B,8h,8w,2]. */
int rb_upsample_convex(const float* coords1, const float* mask, float* out, int B, int h, int w,
                       void* stream);
/* scale = 1.0 reproduces the reference (no x8, utils.py:110); upstream RAFT would pass 8.0. */
int rb_upflow8(const float* coords1, float* out, int B, int h, int w, float scale, void* stream);
/* Cropped forms: out is [B,out_h,out_w,2] = rows [top, top+out_h) x cols [left, left+out_w) of the 8h x 8w field
 * (frames that rb_frames_prepare padded to a multiple of 8 are cropped back by the upsampling kernel itself). */
int rb_upsample_convex_crop(const float* coords1, const float* mask, float* out, int B, int h, int w,
                            int top, int left, int out_h, int out_w, void* stream);
int rb_upflow8_crop(const float* coords1, float* out, int B, int h, int w, float scale, int top, int left,
                    int out_h, int out_w, void* stream);

/* ---- F3 (input edge): dataflow/test_dataflow.py:56-61,96-97 + the SURVEY 8(d) shape policy ------------------
 * src: [B,H,W,3] device frames, BGR like cv2.imdecode -- fp32 in [0,1] (src_is_u8 = 0) or uint8 in [0,255]
 * (src_is_u8 = 1: x/255.0f, the reference's np.float32(x)/255.0, bit for bit).  dst: [B,H+pt+pb,W+pl+pr,3] fp32
 * in [0,1], replicate-padded (upstream InputPadder; the caller chooses the split).  The 2x-1 of
 * RAFT.input_preprocess (RAFT.py:53-59) is applied inside rb_encoder_forward. */
int rb_frames_prepare(const void* src, int src_is_u8, float* dst, int B, int H, int W, int pad_top,
                      int pad_bottom, int pad_left, int pad_right, void* stream);

/* ---- F5 (output edge): forward-backward consistency (occlusion) check, both directions in one launch -----------
 * flow_fw, flow_bw: [B,H,W,2] fp32 (x, y), 8-byte aligned; occ_fw, occ_bw: [B,H,W] uint8.  Displacements are scale*flow
 * pixels (8.0 for raft-small's flow, which keeps the reference's missing x8 of upflow8, utils.py:105-111; 1.0 for
 * raft-things).  For each direction with flow f and the other direction's flow g, at pixel p: u = scale*f(p), t = p + u;
 * occ = 2 if t lies outside [0,W-1] x [0,H-1]; else g' = scale*bilinear(g, t) (corners floor(t) and min(floor(t)+1, dim-1))
 * and occ = 1 if |u + g'|^2 >= alpha1 (|u|^2 + |g'|^2) + alpha2, otherwise 0 (Sundaram et al. 2010, UnFlow).
 * scale > 0, alpha1 >= 0, alpha2 >= 0. */
int rb_flow_consistency(const float* flow_fw, const float* flow_bw, uint8_t* occ_fw, uint8_t* occ_bw, int B, int H,
                        int W, float scale, float alpha1, float alpha2, void* stream);

/* ---- F1: BasicEncoder / SmallEncoder  networks/model_utils.py:61-105 (+ input_preprocess RAFT.py:53-59) --
 * norm: 0 = 'none', 1 = 'instance' (fnet), 2 = 'batch' (cnet of raft-things; folded into the convs at pack
 * time from inference statistics).  Convs are enumerated in execution order; names are relative to the
 * encoder scope ("conv1", "layer2/0/downsample.0", ...), rb_encoder_norm_name gives the scope of the norm
 * that follows conv i ("" = none).  W_host[i] HWIO fp32, b_host[i] [cout]; bn_host[i] (norm == 2 only) is
 * [gamma | beta | mean/EMA | variance/EMA], 4*cout floats.  image: [B,H,W,3] fp32 in [0,1] (2x-1 is applied
 * inside); out: [B,ceil(H/8),ceil(W/8),out_dim] fp32.  The workspace must be zero-filled once before first use. */
int rb_encoder_num_convs(int small);
const char* rb_encoder_conv_name(int small, int i);
const char* rb_encoder_norm_name(int small, int i);
int rb_encoder_conv_shape(int small, int i, int out_dim, int* k, int* stride, int* cin, int* cout);
int rb_encoder_weights_bytes(int small, int out_dim, size_t* bytes);
int rb_encoder_weights_pack(int small, int norm, int out_dim, const float* const* W_host,
                            const float* const* b_host, const float* const* bn_host, void* blob,
                            size_t blob_bytes, void* stream);
/* Host-only forms (no GPU needed), as for the update block; conv index i as in rb_encoder_conv_name.  The stem is packed
 * as a 4x1 conv over the space-to-depth view (csrc/encoder.cu), batch norm is folded into weights and bias. */
int rb_encoder_weights_pack_host(int small, int norm, int out_dim, const float* const* W_host, const float* const* b_host,
                                 const float* const* bn_host, void* host_blob, size_t blob_bytes);
int rb_encoder_packed_conv(int small, int out_dim, int i, size_t* hi_off, size_t* lo_off, size_t* bias_off, int* kh, int* kw,
                           int* cin_pad, int* cout_pad);
int rb_encoder_workspace_bytes(int small, int B, int H, int W, size_t* bytes);
int rb_encoder_forward(int small, int norm, const void* weights, const float* image, float* out, int B,
                       int H, int W, int out_dim, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RAFT_B200_H_ */
