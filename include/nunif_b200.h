/*
 * nunif_b200 - C ABI of the B200-native engine for nunif's two hot paths.
 *
 * The reference (nagadomi/nunif) is pure Python; it has no FFI.  The boundary a
 * maintainer binds is therefore "one C entry point per reference callable on
 * the hot path" (SURVEY.md section 8b).  Each declaration cites the reference
 * callable it replaces (paths relative to nagadomi/nunif @ d23721f).  The
 * ctypes binding the reference would add is shown in INTEGRATION.md and
 * implemented in nunif_b200/_lib.py.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host
 *   - images are planar float32 CHW / BCHW exactly as the reference passes them
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream)
 *   - divergence / convergence are doubles: the reference folds them into fp32 constants from
 *     Python floats (e.g. float(shift_size * convergence)), and bit-exactness needs the same rounding
 *   - every function returns 0 on success, non-zero on error;
 *     nb200_last_error() returns a thread-local message
 *   - there is no CPU fallback: a call without a usable sm_100 device fails
 */
#ifndef NUNIF_B200_H
#define NUNIF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NB200_ABI_VERSION 1

const char* nb200_last_error(void);
int nb200_abi_version(void);
/* device 0..n-1 must be compute capability 10.x; returns non-zero otherwise */
int nb200_check_device(int device);
/* number of kernels this library has launched in this process (bench `gpu_launches`) */
uint64_t nb200_launch_count(void);

/* ------------------------------------------------------------------ *
 * Path A: tiled render (nunif/utils/seam_blending.py)
 * ------------------------------------------------------------------ */

typedef struct nb200_tile_config {
    /* SeamBlending.create_config, seam_blending.py:109-143 */
    int32_t y_h, y_w, h_blocks, w_blocks;
    int32_t pad_l, pad_r, pad_t, pad_b;
    int32_t y_buffer_h, y_buffer_w;
    int32_t input_tile_step, output_tile_step;
} nb200_tile_config;

/* host-side integer planner; bit-exact with the reference. */
int nb200_tile_config_create(int x_h, int x_w, int scale, int offset, int tile_size,
                             int blend_size, nb200_tile_config* out_host);

/* seam_blending.py:82-92: replicate-pad + unfold of tiles [tile0, tile0+n) in raster
 * order into an NHWC fp16 tile batch  dst[n][T][T][cpad]  (channels >= C zero). */
int nb200_tile_unfold(const float* x, int C, int H, int W, const nb200_tile_config* cfg_host,
                      int tile_size, int tile0, int n, void* dst_nhwc_f16, int cpad, void* stream);

/* seam_blending.py:156-174 (update) + :39-40 (get_output) in closed form:
 *   out[C][y_h][y_w] = clamp( sum_t w_t*z_t / sum_t w_t , 0, 1 )
 * over the (at most 4) tiles covering each output pixel, summed in raster tile order.
 * z_all: fp16 planar [h_blocks*w_blocks][C][S][S], S = tile_size*scale - 2*offset.
 * w = create_blend_filter (seam_blending.py:146-153) evaluated in closed form;
 * blend_size==0 reproduces the plain store of :173. */
int nb200_tile_gather_blend(const void* z_all_f16, int C, const nb200_tile_config* cfg_host,
                            int scale, int offset, int tile_size, int blend_size,
                            float* out, void* stream);

/* ------------------------------------------------------------------ *
 * Path A: models.  A model handle owns packed fp16 weights on one device.
 * ------------------------------------------------------------------ */

typedef struct nb200_model nb200_model;

enum {
    NB200_MODEL_UPCUNET = 1,        /* waifu2x.upcunet  (waifu2x/models/cunet.py:139-170) */
    NB200_MODEL_CUNET = 2,          /* waifu2x.cunet    (cunet.py:173-203)                */
    NB200_MODEL_SWIN_UNET_1X = 3,   /* waifu2x.swin_unet_1x (swin_unet.py:208-226)        */
    NB200_MODEL_SWIN_UNET_2X = 4,   /* waifu2x.swin_unet_2x (swin_unet.py:229-251)        */
    NB200_MODEL_SWIN_UNET_4X = 5,   /* waifu2x.swin_unet_4x (swin_unet.py:261-303)        */
    /* Depth-Anything-V2 ViT-S: third-party net the reference loads through torch.hub
     * (iw3/depth_anything_model.py:223-230); state_dict keys `pretrained.*`, `depth_head.*` */
    NB200_MODEL_DEPTH_ANYTHING_V2_S = 6,
    NB200_MODEL_ROW_FLOW_V3 = 7,    /* sbs.row_flow_v3, iw3's default learned stereo warp (iw3/models/row_flow_v3.py) */
    NB200_MODEL_DEPTH_ANYTHING_V2_B = 8,   /* Any_V2_B: ViT-B encoder, 128 head features */
    NB200_MODEL_DEPTH_ANYTHING_V2_L = 9,   /* Any_V2_L: ViT-L encoder (24 blocks), 256 head features */
    NB200_MODEL_DEPTH_AA = 10,             /* iw3.depth_aa, learned anti-aliasing of the depth map (iw3/models/depth_aa.py) */
    NB200_MODEL_MLBW = 11,                 /* sbs.mlbw, multi-layer learned stereo warp, num_layers 2 | 4 (iw3/models/mlbw.py) */
    /* ZoeD_N metric depth: third-party net the reference loads through torch.hub "nagadomi/ZoeDepth_iw3" (iw3/zoedepth_model.py:151-157);
     * state_dict keys of ZoeD_M12_N.pt (`core.core.pretrained.*`, `core.core.scratch.*`, `conv2`, `seed_bin_regressor`, ...).
     * The widths are read off the tensor sizes (BEiT-L/16 for the released checkpoint). */
    NB200_MODEL_ZOEDEPTH_N = 12
};

/* Create a model from named fp32 host tensors using the reference's state_dict
 * keys (nunif/models/utils.py:42-74 load_model / load_state_dict).
 * names[i] is the key, data_host[i] a contiguous float32 buffer of numel[i]
 * elements.  Missing/extra keys are an error, like strict load_state_dict. */
int nb200_model_create(int kind, int n_tensors, const char* const* names,
                       const float* const* data_host, const int64_t* numel,
                       int no_clip, nb200_model** out);
void nb200_model_destroy(nb200_model* m);
/* i2i contract of nunif/models/model.py:65-86 */
int nb200_model_info(const nb200_model* m, int* scale, int* offset, int* blend_size);
/* raw packed weight blob (for the one-time NCCL broadcast that replaces
 * torch.nn.parallel.replicate, nunif/models/data_parallel.py:16,58) */
int nb200_model_weight_blob(nb200_model* m, void** dev_ptr, size_t* bytes);

/* model(minibatch) of seam_blending.py:94-95 under autocast fp16:
 * x: NHWC fp16 [n][T][T][8] (from nb200_tile_unfold, channels 3..7 zero)
 * z: planar [n][3][S][S], S = T*unet_scale/downscale - 2*offset; fp16 for downscale == 1 (the reference's model
 *    output is fp16 under autocast as well), fp32 for downscale 2 | 4 (SwinUNetDownscaled resizes z.float() and
 *    returns fp32, waifu2x/models/swin_unet.py:366-379).
 * downscale in {1,2,4}: 2/4 apply SwinUNetDownscaled (swin_unet.py:366-379). */
int nb200_model_forward(nb200_model* m, const void* x_nhwc_f16, int n, int tile_size,
                        int downscale, void* z_f16, void* stream);

/* nunif.utils.render.tiled_render (render.py:8-19): whole image, device pointers. */
int nb200_tiled_render(nb200_model* m, const float* x, int C, int H, int W, int tile_size,
                       int batch_size, int downscale, float* out, void* stream);

/* The same render with HOST buffers (planar fp32, pinned for full overlap): one H2D copy of the
 * frame, then the output is blended and copied back in bands of finished tile rows on a side
 * stream while later tile batches compute.  `stream` completes after the last band has landed
 * in out_host.  This is the entry point a non-torch binding uses (INTEGRATION.md) and the one
 * bench.py's e2e figure times.  Replaces the host<->device hops around
 * Waifu2x.render (waifu2x/utils.py:218-243; SeamBlending.tiled_render moves each minibatch with .to(device),
 * seam_blending.py:94). */
int nb200_tiled_render_host(nb200_model* m, const float* x_host, int C, int H, int W, int tile_size,
                            int batch_size, int downscale, float* out_host, void* stream);

/* DepthAnythingV2.forward as called by DepthAnythingModel._forward (iw3/depth_anything_model.py:113-119):
 * x [B][3][H][W] fp32, ImageNet-normalised (nb200_da_preprocess), H and W multiples of 14
 * -> depth [B][H][W] fp32 (relative inverse depth, larger = nearer). */
int nb200_depth_anything_forward(nb200_model* m, const float* x, int B, int H, int W, float* depth,
                                 void* stream);

/* ZoeDepth.forward(x)['metric_depth'] as called by zoedepth_model._forward (iw3/zoedepth_model.py:23-27):
 * x [B][3][H][W] fp32, normalised (x - 0.5) / 0.5 and reflection padded (nb200_zoe_preprocess), H and W multiples of 32
 * -> depth [B][H][W] fp32 (metric depth, larger = farther; batch_infer negates it, zoedepth_model.py:124-130). */
int nb200_zoedepth_forward(nb200_model* m, const float* x, int B, int H, int W, float* depth, void* stream);
/* Host-only helper of the same path: the per-block relative-position table ((2g-1)^2 + 3 rows x heads, learned on a g x g token
 * grid) resampled for a ph x pw grid as MiDaS backbones/beit.py `_get_rel_pos_bias` does (bilinear, the 3 class-token rows kept). */
int nb200_zoe_rel_pos_table(const float* table, int g, int heads, int ph, int pw, float* out);

/* iw3.depth_aa (iw3/models/depth_aa.py:46-87; applied by batch_infer when depth_aa is set, iw3/depth_anything_model.py:153-154):
 * x [B][1][H][W] fp32 -> out, same shape.  mode 0 = forward in eval mode (clamp to [0,1]), 1 = infer (normalise by the
 * min / max of the WHOLE tensor, filter without clamp, de-normalise), 2 = forward(clamp=False). */
int nb200_depth_aa(nb200_model* m, const float* x, int B, int H, int W, int mode, float* out, void* stream);

/* sbs.row_flow_v3 in delta_output mode (iw3/models/row_flow_v3.py:57-68,111-116): x [B][3][h][w] fp32 = depth,
 * divergence feature, convergence feature (make_input_tensor, iw3/backward_warp.py:18-63) -> delta [B][1][h][w]
 * fp32 (the x component; the y component is zero). */
int nb200_row_flow_delta(nb200_model* m, const float* x, int B, int h, int w, float* delta, void* stream);

/* sbs.mlbw in delta_output mode (iw3/models/mlbw.py:96-127,237-245): x [B][3][h][w] fp32 (depth, divergence feature,
 * convergence feature) -> delta [B][L][h][w] (x component of each flow layer) and layer_weight [B][L][h][w] (softmax over
 * the L layers); L = nb200_mlbw_num_layers (2 or 4, read off the state_dict).  hole_mask models are not supported. */
int nb200_mlbw_delta(nb200_model* m, const float* x, int B, int h, int w, float* delta, float* layer_weight, void* stream);
int nb200_mlbw_num_layers(const nb200_model* m);

/* backward_warp(c, grid, delta, delta_scale) of the learned warps (iw3/backward_warp.py:67-83,213-226):
 * c [B][3][H][W], delta [B][1][h][w] fp32 -> out [B][3][H][W] = clamp(grid_sample(c, grid + delta*delta_scale)). */
int nb200_backward_warp_delta(const float* c, const float* delta, int B, int H, int W, int h, int w,
                              double delta_scale, float* out, void* stream);

/* AlphaBorderPadding.forward (nunif/utils/alpha.py:32-57): rgb [3][H][W], alpha [1][H][W] fp32 ->
 * out [3][H][W]: transparent pixels are filled from their opaque neighbours, `offset` rounds
 * (offset = the model's i2i_offset, waifu2x/utils.py:271), then clamped to [0,1]. */
size_t nb200_alpha_border_padding_workspace(int H, int W);
int nb200_alpha_border_padding(const float* rgb, const float* alpha, int H, int W, int offset,
                               float* out, void* workspace, void* stream);

/* tta_split (nunif/transforms/tta.py:20-33): view k in 0..7 of x [C][H][W]
 * (identity, hflip, vflip, vflip+hflip, then the same four of rot90) -> out [C][H][W] (k<4)
 * or [C][W][H] (k>=4).  tta_merge (:36-48): views[k] is the render of view k, i.e.
 * [C][H][W] for k<4 and [C][W][H] for k>=4 (H, W = merged size) -> out = clamp(mean of the
 * inverse-transformed views).  `views` is a host array of 8 device pointers. */
int nb200_tta_transform(const float* x, int C, int H, int W, int k, float* out, void* stream);
int nb200_tta_merge(const float* const* views, int C, int H, int W, float* out, void* stream);

/* ------------------------------------------------------------------ *
 * Path B: iw3 depth post-processing and stereo warps
 * ------------------------------------------------------------------ */

enum { NB200_VIEW_BOTH = 0, NB200_VIEW_LEFT = 1, NB200_VIEW_RIGHT = 2 };
enum { NB200_COMPOSE_NONE = 0,      /* separate left/right planar tensors            */
       NB200_COMPOSE_SBS = 1,       /* iw3/utils.py:466-469 cat([L,R], dim=2)+clamp  */
       NB200_COMPOSE_ANAGLYPH_DUBOIS = 2 /* iw3/anaglyph.py:51-92                    */ };

/* iw3/backward_warp.py:96-121 apply_divergence_grid_sample.
 * c: [B][3][H][W], depth: [B][1][h][w] (any resolution).
 * compose NONE: left,right = [B][3][H][W]; SBS: left = [B][3][H][2W], right unused;
 * ANAGLYPH: left = [B][3][H][W], right unused. */
int nb200_backward_warp(const float* c, const float* depth, int B, int H, int W, int h, int w,
                        double divergence, double convergence, int synthetic_view, int compose,
                        float* left, float* right, void* stream);

/* iw3/forward_warp.py:246-256 apply_divergence_forward_warp (inconsistent_shift=False).
 * depth: [B][1][h][w]; if (h,w)!=(H,W) it is resized like forward_warp.py:146-148.
 * fill!=0 <=> method=="forward_fill".  masks may be NULL (return_mask=False).
 * workspace: nb200_forward_warp_workspace() bytes (may be NULL if depth is full-res). */
size_t nb200_forward_warp_workspace(int B, int H, int W, int h, int w);
int nb200_forward_warp(const float* c, const float* depth, int B, int H, int W, int h, int w,
                       double divergence, double convergence, int fill, int synthetic_view,
                       int width_base, int compose, float* left, float* right,
                       float* left_mask, float* right_mask, void* workspace, void* stream);

/* iw3/dilation.py:115-142 dilate_edge(x, [x_iter, y_iter]); x,out: [B][1][h][w];
 * workspace: nb200_dilate_edge_workspace() bytes. */
size_t nb200_dilate_edge_workspace(int B, int h, int w);
int nb200_dilate_edge(const float* x, int B, int h, int w, int x_iter, int y_iter,
                      float* out, void* workspace, void* stream);

/* iw3/depth_scaler.py:4-17 with per-frame amin/amax (base_depth_model.py:176-194)
 * followed by the mapper (iw3/mapper.py:29-32): mapper_c < 0 => "none",
 * else distance_to_disparity(x, mapper_c) (div_6 => 0.6).  In place allowed. */
int nb200_minmax_map(const float* depth, int B, int n_per_frame, float mapper_c,
                     float* out, float* minmax_out /* [B][2] or NULL */, void* stream);

/* Stateful depth normaliser: MinMaxBuffer + EMAMinMaxScaler (iw3/depth_scaler.py:33-142; BaseDepthModel.enable_ema /
 * minmax_normalize_chw / flush_minmax_normalize, iw3/base_depth_model.py:152-194).  All values stay on the device; the
 * host only counts calls, so a frame costs three small launches and no synchronisation (csrc/ema_scaler.cu).
 * mode: 0 = "minmax", 1 = "max".  reset: decay < 0 / buffer_size <= 0 keep the current value (:76-86).
 * update: pushes the frame's amin/amax, *filled = the look-ahead buffer is full, i.e. the OLDEST queued frame can now be
 *   normalised (the frame queue itself lives with the caller).
 * normalize: from_ring = 0 uses the EMA values (:108-116), 1 the ring's amin/amax (flush before a value exists, :127-128);
 *   mapper_c >= 0 applies distance_to_disparity(x, mapper_c) afterwards; minmax_out: optional 2 floats on the device. */
typedef struct nb200_ema_scaler nb200_ema_scaler;
int nb200_ema_scaler_create(int buffer_size, double decay, int mode, nb200_ema_scaler** out);
void nb200_ema_scaler_destroy(nb200_ema_scaler* s);
int nb200_ema_scaler_reset(nb200_ema_scaler* s, double decay, int buffer_size);
int nb200_ema_scaler_update(nb200_ema_scaler* s, const float* frame, int n, int* filled, void* stream);
int nb200_ema_scaler_normalize(nb200_ema_scaler* s, const float* frame, int n, int from_ring,
                               float mapper_c, float* out, float* minmax_out, void* stream);
/* iw3/mapper.py:29-32 get_mapper("div_*") alone: distance_to_disparity(x, mapper_c); in place allowed. */
int nb200_depth_mapper(const float* depth, long long n, float mapper_c, float* out, void* stream);

/* iw3/anaglyph.py:51-92 on already-warped eyes: l,r,out [B][3][H][W] */
int nb200_anaglyph_dubois(const float* l, const float* r, int B, int H, int W, int clip_before,
                          float* out, void* stream);

/* ------------------------------------------------------------------ *
 * Low-level ops (exported for unit tests and micro-benchmarks; the model
 * entry points above are sequences of these)
 * ------------------------------------------------------------------ */

/* F.interpolate(depth, size=(H,W), mode="bilinear", align_corners=True, antialias=True)
 * as used at iw3/forward_warp.py:146-148 (the forward warp fuses this; this entry
 * materialises it). depth [B][1][h][w] -> out [B][1][H][W]. */
int nb200_depth_resize_aa(const float* depth, int B, int h, int w, int H, int W, float* out, void* stream);

/* tcgen05 implicit GEMM on NHWC fp16 activations (csrc/gemm_tcgen05.cuh).
 * kind: 0 linear over flattened pixels, 1 linear with 2-D tiling, 2 conv3x3 valid (4 = conv3x3 zero-padded by 1),
 *       3 conv2x2 stride 2.  Wt: fp16 [N][taps*Cin] with K ordered (ky, kx, c).
 * act: 0 none, 1 LeakyReLU(0.1), 2 GELU(erf), 3 ReLU.
 * out_mode 1: N = 4*cout ordered (dy,dx,co), pixel-shuffle(2) scatter (ConvTranspose2d
 * k2 s2 / Linear+pixel_shuffle).  res: optional residual read at (y+res_cy, x+res_cx). */
int nb200_conv_gemm_f16(const void* A, int B, int Hi, int Wi, int Ci, int Cin, int kind,
                        const void* Wt, int N, const float* bias, int act, void* out, int ldo,
                        int out_mode, int cout, const void* res, int ldr, int res_H, int res_W,
                        int res_cy, int res_cx, int res_before_act, void* stream);

/* shifted-window attention core between the qkv and proj Linears
 * (torchvision swin_transformer.py:166-221), window 6x6, 6 heads.
 * qkv: three dense planes q | k | v, each [B][H][W][C] fp16 (how the engine's qkv GEMM writes them)
 * -> out [B][H][W][C] fp16; bias_table fp32 [121][6]. */
int nb200_window_attention_f16(const void* qkv, const float* bias_table, void* out, int B,
                               int H, int W, int C, int heads, int shift, void* stream);

/* Fused tail of one SwinTransformerBlock (torchvision swin_transformer.py:228 proj, :453-455; MLP = Linear-GELU-Linear,
 * ratio 2, Identity norms: waifu2x/models/swin_unet.py:16-17,31), one tcgen05 kernel (csrc/swin_fused_mlp.cu):
 *   x1 = x + att @ wp^T + bp   (att == NULL: x1 = x);   x <- x1 + gelu(x1 @ w1^T + b1) @ w2^T + b2
 * x, att: [T][C] fp16 (x updated in place); wp [C][C], w1 [2C][C], w2 [C][2C] fp16; biases fp32.  C in {96, 192}. */
int nb200_swin_mlp_fused_f16(void* x, const void* att, long long T, int C, const void* wp,
                             const float* bp, const void* w1, const float* b1, const void* w2,
                             const float* b2, void* stream);

/* Fused head of one SwinTransformerBlock: qkv Linear + shifted 6x6 window attention (swin_transformer.py:166-221;
 * everything but the proj Linear), one kernel (csrc/swin_fused_attn.cu): the qkv GEMM runs on tcgen05, q/k/v stay in
 * shared memory.  x, att: [B][H][W][C] fp16; wqkv [3C][C] fp16 and bqkv [3C] fp32 in the reference's row order
 * (q | k | v); bias_table fp32 [121][6] (relative_position_bias_table).  C in {96, 192}, 6 heads. */
int nb200_swin_attn_fused_f16(const void* x, const void* wqkv, const float* bqkv,
                              const float* bias_table, void* att, int B, int H, int W, int C,
                              int shift, void* stream);
/* The same operator and operands with QK^T and PV on tcgen05 as well (csrc/swin_attn_tc.cu: S and P live in tensor
 * memory / shared memory, three windows per 128-row UMMA); this is the kernel the model path launches. */
int nb200_swin_attn_tc_f16(const void* x, const void* wqkv, const float* bqkv,
                           const float* bias_table, void* att, int B, int H, int W, int C,
                           int shift, void* stream);

/* Frame-edge conversions (nunif/utils/video.py:218-223 to_tensor, :236-246 from_tensor,
 * iw3/utils.py:274-289 hwc_to_chw_float): x [B][H][W][3] uint8 (bits=8) or uint16 (bits=16)
 * <-> [B][3][H][W] fp32 in [0,1]; the fp32 -> integer direction rounds half to even. */
int nb200_hwc_to_chw_f32(const void* x, int bits, int B, int H, int W, float* out, void* stream);
int nb200_chw_f32_to_hwc(const float* x, int bits, int B, int H, int W, void* out, void* stream);

/* DepthAnything batch_preprocess (iw3/depth_anything_model.py:69-110): size rule (host,
 * integers) and the fused antialiased-bilinear resize + clamp + ImageNet normalise:
 * x [B][3][H][W] fp32 in [0,1] -> out [B][3][new_h][new_w] fp32. */
int nb200_da_preprocess_size(int H, int W, int lower_bound, int max_aspect_ratio,
                             int limit_resolution, int* new_h, int* new_w);
int nb200_da_preprocess(const float* x, int B, int H, int W, int new_h, int new_w, float* out,
                        void* stream);

/* ZoeDepth batch_preprocess (iw3/zoedepth_model.py:30-85): size rule (host integers) and the fused
 * antialiased resize + reflection pad (nunif/modules/reflection_pad2d.py:57-68) + clamp + normalise:
 * x [B][3][H][W] -> out [B][3][frame_h + 2*pad_h][frame_w + 2*pad_w] (== new_h x new_w in landscape). */
int nb200_zoe_preprocess_size(int H, int W, int h_height, int v_height, int mod, int* new_h,
                              int* new_w, int* pad_h, int* pad_w, int* frame_h, int* frame_w);
int nb200_zoe_preprocess(const float* x, int B, int H, int W, int frame_h, int frame_w, int pad_h,
                         int pad_w, float* out, void* stream);

/* iw3/anaglyph.py:95-110 apply_anaglyph_redcyan: l, r [B][3][H][W] fp32 -> out [B][3][H][W]. */
enum { NB200_ANAGLYPH_DUBOIS = 0, NB200_ANAGLYPH_DUBOIS2 = 1, NB200_ANAGLYPH_COLOR = 2, NB200_ANAGLYPH_GRAY = 3,
       NB200_ANAGLYPH_HALF_COLOR = 4, NB200_ANAGLYPH_WIMMER = 5, NB200_ANAGLYPH_WIMMER2 = 6 };
int nb200_anaglyph(const float* l, const float* r, int B, int H, int W, int type, float* out, void* stream);

/* TF.resize(x, (oh, ow), BICUBIC, antialias=True) on `planes` fp32 H x W planes (half-SBS / half-TB and the
 * max-output-size resize of postprocess_image, iw3/utils.py:445-485); clamp01_out applies the following clamp. */
int nb200_resize_bicubic_aa(const float* x, int planes, int H, int W, int oh, int ow, int clamp01_out,
                            float* out, void* stream);

/* VR180 output (iw3/equirectangular.py:7-40; iw3/utils.py:441-443): zero-pad to 1.5 x the longer edge, bicubic grid_sample
 * (zeros, align_corners=True) through x' = k tan(az), y' = k tan(el)/cos(az), clamp [0,1].
 * c [C][H][W] -> out [C][out_h][out_w] with (out_h, out_w) from nb200_equirectangular_size (host rule). */
int nb200_equirectangular_size(int H, int W, int* out_h, int* out_w);
int nb200_equirectangular(const float* c, int C, int H, int W, float* out, void* stream);

/* Kernel-class device timing (CUDA events around every launch of this library) used by
 * bench.py for the live roofline figure.  report writes a JSON object
 * {"gemm": {"launches": n, "ms": t, "work": flops_or_bytes}, ...} and synchronises the device. */
int nb200_tune_set(int key, int value);   /* GEMM scheduling knobs for profiles/gemm_bench.py */
int nb200_debug_tap(int id, void* dev_buf, size_t capacity);  /* copy intermediate `id` of nb200_zoedepth_forward to dev_buf (profiles/debug_zoe.py) */
int nb200_debug_timeline(void* dev_buf);  /* per-role clock64 timeline of CTA 0 (profiles/gemm_timeline.py) */
int nb200_profile_enable(int on);
int nb200_profile_report(char* buf, size_t cap);
int nb200_profile_dump(char* buf, size_t cap);   /* one CSV line per timed launch: class,ms,work,read_bytes,write_bytes */

/* ------------------------------------------------------------------ *
 * Low-level ops of the depth networks, exposed for unit tests
 * (csrc/depth_kernels.cu, csrc/zoe_kernels.cu; the Depth-Anything-V2 and
 * ZoeD_N forwards above are sequences of these and the GEMM)
 * ------------------------------------------------------------------ */

/* dinov2 Attention / BEiT attention core: softmax(q k^T / 8 [+ bias]) v per image and head, head dim 64.
 * qkv fp16 [B*N][3*heads*64] (q | k | v, head-major) -> out fp16 [B*N][heads*64].  bias_log2e (may be NULL): fp32
 * [heads][N][ldb] already multiplied by log2 e, shared by the B images; ldb even and >= cdiv(N, 64) * 64. */
int nb200_vit_attention_f16(const void* qkv, void* out, int B, int N, int heads, const float* bias_log2e, int ldb,
                            void* stream);
/* residual add + LayerNorm(eps=1e-6) of the ViT blocks: x32 fp32 [rows][dim] += fp16 delta (may be NULL);
 * out fp16 [rows][dim] = LayerNorm(x32) * w + b (out NULL: only the residual is updated).  dim in {256, 384, 768, 1024}. */
int nb200_vit_add_layernorm(float* x32, const void* delta, const float* w, const float* b, void* out, long long rows,
                            int dim, void* stream);
/* MiDaS beit.py gen_relative_position_index gather: bias[h][q][k] (row stride ldb >= N, N = ph*pw + 1) =
 * table[index(q, k)][h] * log2 e; table fp32 [(2ph-1)(2pw-1) + 3][heads].  Columns [N, ldb) are not written. */
int nb200_zoe_expand_rel_bias(const float* table, int ph, int pw, int heads, float* bias, int ldb, void* stream);
/* ZoeDepth AttractorLayerUnnormed (softplus attractors, align-corners bilinear prev_bin, inv_attractor mean):
 * apre fp16 [B*H*W][lda] (first na used), prev_bin fp32 [B][h][w][64] -> out fp32 [B][H][W][64]. */
int nb200_zoe_attractor(const void* apre, int lda, int na, const float* prev_bin, int B, int h, int w, int H, int W,
                        float* out, void* stream);
/* ZoeDepth ConditionalLogBinomial tail + sum_k prob_k * centre_k: g fp16 [B*H*W][ldg >= 80] (GELU'd hidden), w2 fp32
 * [4][80], b2 [4], bins fp32 [B][h][w][64] (align-corners bilinear to H x W) -> depth fp32 [B][H][W]. */
int nb200_zoe_clb_final(const void* g, int ldg, const float* w2, const float* b2, const float* bins, int B, int h, int w,
                        int H, int W, float* depth, void* stream);
/* F.interpolate(x, (H, W), mode="bilinear", align_corners=True) of the DPT head on fp16 NHWC:
 * x [B][h][w][C] -> out [B][H][W][C], C % 8 == 0. */
int nb200_dpt_upsample_bilinear_f16(const void* x, int B, int h, int w, int C, void* out, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NUNIF_B200_H */
