/*
 * r3dp_b200.h — C ABI of libr3dp_b200.so: the B200 (sm_100a) implementation of Real3D-Portrait's per-frame
 * volumetric render + super-resolution hot path.
 *
 * The reference has no C ABI for this path: its boundary is Python `torch.nn.Module.forward` signatures
 * (SURVEY.md §8b).  The host-side mirror of those signatures lives in `real3dportrait_b200/*.py` and binds THIS
 * header through ctypes; each entry point below names the reference interface it stands behind (paths relative
 * to the reference tree).  Conventions:
 *   - every pointer is a DEVICE pointer on the current CUDA device unless the name ends in `_host`;
 *   - tensors are dense row-major fp32 unless stated; shapes are given in brackets;
 *   - `stream` is a cudaStream_t (0 = legacy default stream); all work is enqueued asynchronously on it and
 *     nothing synchronises the device;
 *   - return value 0 = success, non-zero = error; `r3dp_last_error()` returns a thread-local message
 *     (the Python mirror raises RuntimeError with it, like the reference's TORCH_CHECK in bias_act.cpp:39-55);
 *   - inputs are never written; outputs / workspaces must not alias inputs.
 * There is no CPU fallback anywhere behind this ABI.
 */
#ifndef R3DP_B200_H
#define R3DP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define R3DP_ABI_VERSION 2

typedef void* r3dp_stream_t; /* cudaStream_t */

/* OSGDecoder parameters (modules/img2plane/triplane.py:122-146; FullyConnectedLayer networks_stylegan2.py:99-131).
 * Raw (unscaled) state_dict tensors; the 1/sqrt(fan_in) weight gains are applied by the library. */
typedef struct r3dp_mlp {
    const float* w1; /* net.0.weight [hidden, in_features]      */
    const float* b1; /* net.0.bias   [hidden]                   */
    const float* w2; /* net.2.weight [1 + out_dim, hidden]      */
    const float* b2; /* net.2.bias   [1 + out_dim]              */
    int in_features; /* 32 */
    int hidden;      /* 64 */
    int out_dim;     /* 32 (colour channels; +1 density)        */
} r3dp_mlp_t;

int         r3dp_abi_version(void);
const char* r3dp_last_error(void);
/* SM count and compute capability of the current device; fails unless it is sm_100. */
int r3dp_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Running total of CUDA kernels this library has launched in the process (bench.py's `gpu_launches`). */
unsigned long long r3dp_launch_count(void);
/* A/B switches for profiling runs (same meaning as the R3DP_* environment variables, settable at run time):
 *   "render": 0 = streaming kernel for single-pass renders (default), 1 = CTA-per-ray-tile kernel;  "rs_d": 4 | 8 | 16 samples per ray and tile;
 *   "rs_prefetch": frames of planes the fused render streams DRAM -> L2 ahead of its gather (default 2, 0 = off) */
int r3dp_set_option(const char* key, int value);
/* Frame exchange of a sharded clip (inference/real3d_infer.py:515-521 collects the frames of a clip on one device): copy-engine peer copy of
 * `bytes` from `src` on device `src_device` to `dst` on device `dst_device` (e.g. a CUDA-IPC mapping of rank 0's clip buffer), enqueued on
 * `stream` (a stream of the CALLING device); no SM is used and nothing is synchronised. */
int r3dp_peer_copy(void* dst, int dst_device, const void* src, int src_device, size_t bytes, r3dp_stream_t stream);

/* ---------------------------------------------------------------------------------------------------- rays ---
 * RaySampler.forward (modules/eg3ds/volumetric_rendering/ray_sampler.py:24-63).
 * cam2world [N,4,4], intrinsics [N,3,3]  ->  ray_o [N,res*res,3], ray_d [N,res*res,3]; ray m = row*res + col. */
int r3dp_gen_rays(const float* cam2world, const float* intrinsics, int N, int res, float* ray_o, float* ray_d,
                  r3dp_stream_t stream);

/* -------------------------------------------------------------------------------------------------- planes ---
 * Layout change done once per frame before sampling: reference tri-planes are [N,3,C,H,W]
 * (secc_img2plane.py:105-110); the gather kernels read channels-last [N,3,H,W,C] so one bilinear tap is one
 * 128-byte line.  C must be 32. */
int r3dp_planes_to_channels_last(const float* planes_nchw, int N, int C, int H, int W, float* planes_cl,
                                 r3dp_stream_t stream);

/* Tri-grids (`triplane_feature_type: trigrid | trigrid_v2`): grids_nchw [N,3,C*D,H,W] with channel index c*D + d (the reference views
 * it as [N*3,C,D,H,W], renderer.py:83) -> grids_cl [N,3,D,H,W,C]: every depth slice a channels-last plane.  D = 1 is the call above. */
int r3dp_grids_to_channels_last(const float* grids_nchw, int N, int C, int D, int H, int W, float* grids_cl, r3dp_stream_t stream);
/* sample_from_trigrids (renderer.py:78-89): grids_cl [N,3,D,H,W,C], coords [N,P,3] -> out [N,3,P,C]; trilinear, zero padding,
 * align_corners=False; plane p is sampled at (x,y,z), (x,z,y), (z,x,y) x 2/box_warp.  D >= 2. */
int r3dp_trigrid_sample(const float* grids_cl, int N, int C, int D, int H, int W, const float* coords, int P, float box_warp,
                        float* out, r3dp_stream_t stream);
/* r3dp_run_model for tri-grids [N,3,D,H,W,C] (D = 1: tri-planes). */
int r3dp_run_model_grid(const float* planes_cl, int N, int C, int D, int H, int W, const float* coords, int P, float box_warp,
                        const r3dp_mlp_t* mlp, float* rgb, float* sigma, r3dp_stream_t stream);

/* sample_from_planes (renderer.py:65-75): planes_cl [N,3,H,W,C], coords [N,P,3] -> out [N,3,P,C]
 * (bilinear, zero padding, align_corners=False, coords scaled by 2/box_warp; plane axes of generate_planes()). */
int r3dp_triplane_sample(const float* planes_cl, int N, int C, int H, int W, const float* coords, int P,
                         float box_warp, float* out, r3dp_stream_t stream);

/* ImportanceRenderer.run_model (renderer.py:169-188) with an OSGDecoder: gather + mean over planes + MLP.
 * -> rgb [N,P,out_dim], sigma [N,P,1]. */
int r3dp_run_model(const float* planes_cl, int N, int C, int H, int W, const float* coords, int P, float box_warp,
                   const r3dp_mlp_t* mlp, float* rgb, float* sigma, r3dp_stream_t stream);

/* OSGDecoder.forward (modules/img2plane/triplane.py:133-146) on caller-supplied features:
 * feat [N,K,P,C], K = 3 (mean over the planes) or K = 1 (already aggregated) -> rgb [N,P,out_dim], sigma [N,P,1]. */
int r3dp_decode(const float* feat, int N, int K, int P, int C, const r3dp_mlp_t* mlp, float* rgb, float* sigma,
                r3dp_stream_t stream);

/* -------------------------------------------------------------------------------------------------- render ---
 * ImportanceRenderer.forward with ray_start = ray_end = 'auto' (renderer.py:118-167), fused: box limits
 * (math_utils.py:46-98) -> stratified depths (renderer.py:209-232) -> tri-plane gather -> OSGDecoder ->
 * MipRayMarcher2 (ray_marcher.py:25-57) [-> importance resampling (renderer.py:234-297) -> second gather/MLP ->
 * depth merge (renderer.py:197-207) -> final march].
 *   ray_o, ray_d [N,M,3]          rays; if ray_o == NULL they are generated in-kernel from `camera` [N,25]
 *                                 (row-major c2w then row-major K, secc_img2plane.py:95-96) with M = res*res
 *   u_coarse [N,M,S]              the uniforms the reference draws with torch.rand_like (renderer.py:226)
 *   u_fine   [N*M,S_imp] or NULL  the uniforms of torch.rand (renderer.py:281); required when S_imp > 0
 *   res                           image side if the M rays form a res x res image (enables 2-D ray tiles), else 0
 * outputs: rgb [N,M,out_dim] (already scaled to [-1,1]), depth [N,M,1], weights_sum [N,M,1], is_ray_valid [N,M]
 * (uint8 0/1).  Batch-global quirks are reproduced per call: invalid rays inherit min/max of the valid ray starts
 * (renderer.py:123-126) and depth is clamped to the call-wide [min,max] sample depth (ray_marcher.py:50).
 * workspace: r3dp_render_workspace_bytes(N, M) bytes of scratch.
 * Kernels: single-pass renders (S_imp == 0) run the warp-specialised streaming kernel (render_stream.cu: gather, tcgen05 decoder and
 * ray march of consecutive 128-sample tiles overlap inside one persistent CTA per SM); importance renders run the CTA-per-ray-tile
 * kernel (render.cu).  Decoder arithmetic: the OSGDecoder GEMMs run on tcgen05 with every fp32 operand split into two fp16 halves (three
 * partial products, fp32 accumulation in TMEM) - fp32-grade results (rgb within 2e-6 of the CUDA-core decoder); two-pass shapes whose
 * tiles do not fit use the fp32 CUDA-core decoder.  The prepared decoder operands live in the caller's `workspace`, so calls with
 * different decoders may run concurrently on different streams (each with its own workspace).
 * A/B knobs (read once per process): R3DP_RENDER=tile, R3DP_RS_D=4|8|16, R3DP_MLP=tc|smem|const (const keeps process-wide state). */
size_t r3dp_render_workspace_bytes(int N, int M);

/* Channels-last plane addressing, strides in floats: the C = 32 features of texel (plane p, row y, col x) of frame n start at
 *   planes + n*frame_stride + p*plane_stride + y*row_stride + x*texel_stride      (every stride a multiple of 4 floats).
 *   [N,3,H,W,C] (r3dp_planes_to_channels_last)                      plane = H*W*C, row = W*C,   texel = C
 *   [N,H,W,3,C] = the producer's [N,3*C,H,W] conv output held in torch.channels_last memory (secc_img2plane.py:73-81,
 *                 segformer.py:704-733 emit [B,3,C,H,W] views of such a tensor): plane = C, row = W*3*C, texel = 3*C  -> no repack at all
 *   frame_stride = 0: one plane set shared by every frame of the call (the per-clip canonical planes). */
typedef struct r3dp_plane_layout {
    long long frame_stride;
    int plane_stride, row_stride, texel_stride;
    /* tri-grids (`triplane_feature_type: trigrid | trigrid_v2`, sample_from_trigrids, renderer.py:78-89; egs/os_avatar/img2plane.yaml:65-66):
     * every plane is a stack of `depth` >= 2 slices `slice_stride` floats apart, sampled trilinearly with the third projected coordinate
     * (z, y, y for planes 0, 1, 2); depth <= 1: plain tri-planes.  [N,3,D,H,W,C] (r3dp_grids_to_channels_last): slice = H*W*C. */
    int depth, slice_stride;
} r3dp_plane_layout_t;

/* r3dp_render with explicit plane layouts and an optional SECOND plane set sampled at the same points and added to the first
 * (bilinear sampling is linear): `planes = cano_planes + secc_planes` (secc_img2plane.py:73-81) without the 75 MB/frame add. */
typedef struct r3dp_render_args {
    const float* planes;  r3dp_plane_layout_t layout;
    const float* planes2; r3dp_plane_layout_t layout2;   /* NULL = none; strides (except frame_stride) must equal `layout`'s */
    int N, C, H, W;
    const float* ray_o; const float* ray_d; const float* camera; int M, res;
    int S, S_imp; float box_warp; int white_back;
    const float* u_coarse; const float* u_fine;
    const r3dp_mlp_t* mlp;
    float* rgb; float* depth; float* weights_sum; uint8_t* is_ray_valid;
    void* workspace; size_t workspace_bytes;
} r3dp_render_args_t;
int r3dp_render_ex(const r3dp_render_args_t* args, r3dp_stream_t stream);

int r3dp_render(const float* planes_cl, int N, int C, int H, int W,
                const float* ray_o, const float* ray_d, const float* camera, int M, int res,
                int S, int S_imp, float box_warp, int white_back,
                const float* u_coarse, const float* u_fine, const r3dp_mlp_t* mlp,
                float* rgb, float* depth, float* weights_sum, uint8_t* is_ray_valid,
                void* workspace, size_t workspace_bytes, r3dp_stream_t stream);

/* MipRayMarcher2.run_forward (ray_marcher.py:25-57) stand-alone: colors [N,M,S,C], sigmas [N,M,S,1],
 * depths [N,M,S,1] -> rgb [N,M,C], depth [N,M,1], weights [N,M,S-1,1].  workspace: 16 bytes. */
int r3dp_ray_march(const float* colors, const float* sigmas, const float* depths, int N, int M, int S, int C,
                   int white_back, float* rgb, float* depth, float* weights, void* workspace,
                   r3dp_stream_t stream);

/* ------------------------------------------------------------------------------------- super-resolution ---
 * Building blocks of SuperresolutionHybrid8XDC.forward (modules/eg3ds/models/superresolution.py:331-359) with
 * noise_mode='none', fp32 parameters.  Activations are NCHW fp32 at the boundary.
 *
 * r3dp_sr_styles: FullyConnectedLayer(w_dim, Cin, bias_init=1) (networks_stylegan2.py:113-127,314):
 *   styles[N,Cin] = w_lat[N,w_dim] @ (A[Cin,w_dim]/sqrt(w_dim))^T + a[Cin], then * post_scale
 *   (post_scale = 1/sqrt(Cin) for ToRGB, networks_stylegan2.py:362,366).
 * r3dp_sr_fold_weights: the per-sample weights of modulated_conv2d (networks_stylegan2.py:63-70):
 *   wf[N,O,I,k,k] = W[O,I,k,k] * styles[N,I]  (* rsqrt(sum_{I,k,k} (.)^2 + 1e-8) if demodulate). */
int r3dp_sr_styles(const float* w_lat, const float* affine_w, const float* affine_b, int N, int w_dim, int Cin,
                   float post_scale, float* styles, r3dp_stream_t stream);
int r3dp_sr_fold_weights(const float* weight, const float* styles, int N, int O, int I, int k, int demodulate,
                         float* wf, r3dp_stream_t stream);

/* F.interpolate(size, bilinear, align_corners=False, antialias=True) for UP-scaling (superresolution.py:351-355;
 * antialias is the identity when scale >= 1).  x [N,C,h,w] -> y [N,C,size,size]. */
int r3dp_sr_resize_bilinear(const float* x, int N, int C, int h, int w, int size, float* y, r3dp_stream_t stream);

/* Exact-fp32 SynthesisLayer (networks_stylegan2.py:322-342 -> conv2d_resample.py:116-138 -> bias_act lrelu):
 *   up == 1: y = lrelu(conv3x3(x, wf[n], pad 1) + bias) * sqrt(2)                       x,y [N,*,H,W]
 *   up == 2: y = lrelu(FIR4x4(conv_transpose2d(x, wf[n]^T, stride 2), pad 1, gain 4) + bias) * sqrt(2)
 *            x [N,I,H,W] -> y [N,O,2H,2W]; scratch holds the (2H+1)x(2W+1) intermediate:
 *            r3dp_sr_layer_scratch_bytes(N,O,H,W) bytes (0 needed for up == 1). */
size_t r3dp_sr_layer_scratch_bytes(int N, int O, int H, int W);
int r3dp_sr_layer_fp32(const float* x, const float* wf, const float* bias, int N, int I, int O, int H, int W, int up,
                       float* y, void* scratch, r3dp_stream_t stream);

/* ToRGB + skip (networks_stylegan2.py:365-370,463-469):
 *   img_out[N,3,H,W] = upsample2d(img_in[N,3,H/2,W/2]) + conv1x1(x[N,I,H,W], wf_rgb[N,3,I]) + bias[3]
 * upsample2d = zero-insert x2, pad (2,1,2,1), FIR [1,3,3,1]^2/64, gain 4 (upfirdn2d.py:317-354).
 * img_in may be NULL (no skip). */
int r3dp_sr_torgb_fp32(const float* x, const float* wf_rgb, const float* bias, const float* img_in, int N, int I,
                       int H, int W, float* img_out, r3dp_stream_t stream);

/* --------------------------------------------------------------- super-resolution on tensor cores (tcgen05) ---
 * Same layers as above as TMA-fed tcgen05 implicit GEMMs: fp16 operands, fp32 accumulation in TMEM, fp32 epilogue.
 * Activations are NHWC fp16 with channels padded to a multiple of 64; weights are the per-sample folded weights
 * (r3dp_sr_fold_weights) packed to fp16 [Nw][9][O][Ipad] with Nw == N (per-sample styles) or 1 (shared styles).
 * Restrictions (met by SuperresolutionHybrid8XDC): W % 128 == 0, Cout % 128 == 0.
 *
 * r3dp_sr_tc_pack_weights  wf fp32 [Nw,O,I,3,3] -> packed fp16
 * r3dp_sr_tc_input         x fp32 NCHW [N,C,h,w] -> bilinear (align_corners=False) to size x size -> NHWC fp16 [N,size,size,Cpad]
 * r3dp_sr_tc_layer         SynthesisLayer (networks_stylegan2.py:322-342): up == 1 -> y [N,H,W,O]; up == 2 -> y [N,2H,2W,O]
 *                          (transposed conv as 4 parity phases + FIR, conv2d_resample.py:116-133); scratch for up == 2:
 *                          r3dp_sr_tc_scratch_bytes(N,O,H,W)
 * r3dp_sr_tc_torgb         ToRGB + upsampled skip of a non-final block -> img fp32 NCHW [N,3,H,W]
 * r3dp_sr_tc_last_layer    last conv (I -> 128) fused with ToRGB + skip: only the image is written (fp32 NCHW [N,3,H,W]);
 *                          wrgb [Nw,3,128], brgb [3], img_prev [N,3,H/2,W/2]. */
int r3dp_sr_tc_pack_weights(const float* wf, int Nw, int O, int I, void* packed_f16, r3dp_stream_t stream);
int r3dp_sr_tc_input(const float* x, int N, int C, int h, int w, int size, void* y_f16, r3dp_stream_t stream);
size_t r3dp_sr_tc_scratch_bytes(int N, int O, int H, int W);
int r3dp_sr_tc_layer(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W,
                     int up, void* y_f16, void* scratch, r3dp_stream_t stream);
int r3dp_sr_tc_torgb(const void* x_f16, const float* wrgb, const float* brgb, const float* img_prev, int N, int Nw, int C,
                     int H, int W, float* img_out, r3dp_stream_t stream);
/* Up layer (up == 2) for SMALL Cin through FIR-composed weights: FIR(conv_transpose(x,w)) = four 3x3 correlations, one per output
 * parity (4x the MACs, but no (2H+1)x(2W+1) intermediate / FIR pass).  pack: wf fp32 [Nw,O,I,3,3] -> fp16 [Nw,36,O,Ipad]. */
int r3dp_sr_tc_pack_weights_up_composed(const float* wf, int Nw, int O, int I, void* packed_f16, r3dp_stream_t stream);
int r3dp_sr_tc_layer_up_composed(const void* x_f16, const void* wpc_f16, const float* bias, int N, int Nw, int I, int O, int H,
                                 int W, void* y_f16, r3dp_stream_t stream);
/* conv3x3 (up == 1) + bias/lrelu -> y fp16 NHWC, fused with the block's ToRGB + upsampled skip -> img_out fp32 NCHW
 * (block0.conv1 + block0.torgb of SynthesisBlock.forward, networks_stylegan2.py:455-469). */
int r3dp_sr_tc_layer_torgb(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                           const float* img_prev, int N, int Nw, int I, int O, int H, int W, void* y_f16, float* img_out,
                           r3dp_stream_t stream);
/* r3dp_sr_tc_input for a channels-last fp32 source [N,h,w,C] (the renderer's [N,M,C] output viewed as an image). */
int r3dp_sr_tc_input_nhwc(const float* x_nhwc, int N, int C, int h, int w, int size, void* y_f16, r3dp_stream_t stream);
/* ... and rgb_out [N,3,size,size] fp32 = the same resize of channels 0..2 (`rgb_image = feature_image[:, :3]`, secc_img2plane.py:126) in the same
 * launch; split != 0 writes the [hi | lo] activation layout of the r3dp_sr_tcx_* path. */
int r3dp_sr_tc_input_nhwc_rgb(const float* x_nhwc, int N, int C, int h, int w, int size, void* y_f16, float* rgb_out, int split, r3dp_stream_t stream);
int r3dp_sr_tc_last_layer(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                          const float* img_prev, int N, int Nw, int I, int H, int W, float* img_out, r3dp_stream_t stream);
/* The same with the caller loop's output conversion fused into the epilogue (inference/real3d_infer.py:515-519):
 *   clamp != 0       img_out clamped to [-1, 1] (imgs.clamp(-1,1))
 *   img_out_u8       non-NULL: write uint8 HWC video frames [N,H,W,3] = uint8(int((clamp(x) + 1) / 2 * 255)) INSTEAD of the fp32 image
 *                    (4x fewer bytes to gather / copy to the host); img_out may then be NULL. */
int r3dp_sr_tc_last_layer_ex(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                             const float* img_prev, int N, int Nw, int I, int H, int W, float* img_out, uint8_t* img_out_u8, int clamp,
                             r3dp_stream_t stream);

/* ---- fp32-grade tensor-core SR (`sr_mode='tc_exact'`): the same layers with SPLIT fp16 operands ------------------------------------------
 * The reference SR computes in fp32 (networks_stylegan2.py:37-94, conv2d_resample.py:48-145).  These entry points keep that accuracy on
 * tcgen05: every fp32 operand is stored as two fp16 halves v = hi + lo (activations NHWC [N,H,W, 2*Cpad] = [hi | lo]; packed weights
 * [Nw,taps,O, 2*Ipad] = [hi | lo] of w * 2^10) and every convolution accumulates hi*hi + lo*hi + hi*lo in fp32 (three times the MMAs; the
 * dropped lo*lo term is ~2^-22).  Same arguments and meaning as the r3dp_sr_tc_* functions of the same name; tensors are twice as wide.
 * Activations are split unscaled, so results are fp32-grade (within 2x of an fp32 evaluation) for layer inputs of magnitude 2^-4 and above;
 * below that the lo halves become fp16 subnormals and the error grows (~1.7e-5 of max|y| at 2^-10, tests/test_cpu_split_conv.py). */
int r3dp_sr_tcx_pack_weights(const float* wf, int Nw, int O, int I, void* packed_f16, r3dp_stream_t stream);
int r3dp_sr_tcx_pack_weights_up_composed(const float* wf, int Nw, int O, int I, void* packed_f16, r3dp_stream_t stream);
int r3dp_sr_tcx_input(const float* x, int N, int C, int h, int w, int size, void* y_f16, r3dp_stream_t stream);
int r3dp_sr_tcx_input_nhwc(const float* x_nhwc, int N, int C, int h, int w, int size, void* y_f16, r3dp_stream_t stream);
size_t r3dp_sr_tcx_scratch_bytes(int N, int O, int H, int W);
int r3dp_sr_tcx_layer(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W,
                      int up, void* y_f16, void* scratch, r3dp_stream_t stream);
int r3dp_sr_tcx_layer_up_composed(const void* x_f16, const void* wpc_f16, const float* bias, int N, int Nw, int I, int O, int H,
                                  int W, void* y_f16, r3dp_stream_t stream);
int r3dp_sr_tcx_layer_torgb(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                            const float* img_prev, int N, int Nw, int I, int O, int H, int W, void* y_f16, float* img_out,
                            r3dp_stream_t stream);
int r3dp_sr_tcx_last_layer(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                           const float* img_prev, int N, int Nw, int I, int H, int W, float* img_out, uint8_t* img_out_u8, int clamp,
                           r3dp_stream_t stream);

/* r3dp_sr_tc_conv with split fp16 operands (x [N,H,W,2*Ipad], weights from r3dp_sr_tcx_pack_weights, y [N,H,W,2*O] = [hi | lo]); used for the small
 * head_torso_alpha_predictor of fuse mode v3, whose output is thresholded (sr_with_ref.py:129-143) and therefore wants fp32-grade arithmetic. */
int r3dp_sr_tcx_conv(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W, int ksize,
                     int act, void* y_f16, r3dp_stream_t stream);

/* Measurement hooks (bench.py): time every tensor-core conv launch with a CUDA-event pair on its launching stream. */
int r3dp_sr_tc_prof(int enable);
int r3dp_sr_tc_prof_read(float* total_ms, int* launches);
/* Debug builds only (-DR3DP_TC_DEBUG_TIMING=1): 32 x 24 uint64 device buffer; row i receives the MMA / epilogue warps' clock sums of the i-th conv launch (NULL = off). */
int r3dp_sr_tc_debug_buffer(void* buf);

/* ------------------------------------------------------- torso head: SuperresolutionHybrid8XDC_Warp building blocks ---
 * (modules/real3d/super_resolution/sr_with_ref.py:16-162; the torso warper itself stays the caller's PyTorch module)
 * r3dp_sr_tc_conv              nn.Conv2d k=1|3, stride 1, same padding (+bias) [+ act: 0 linear, 1 lrelu(0.2)*sqrt2, 2 nn.LeakyReLU 0.01]
 *                              x [N,H,W,Ipad] fp16, weights packed with r3dp_sr_tc_pack_weights (k=1: value in tap 4), y [N,H,W,O] fp16
 * r3dp_sr_tc_layer_torgb_noup  SynthesisBlockNoUp tail: conv3x3 + act -> y, img_out = img_prev (same resolution) + ToRGB(y) + brgb
 * r3dp_sr_alpha_cat            out = cat[xa*alpha, xb*(1-alpha)] on fp16 NHWC (pixel strides stride_a/stride_b in elements), alpha fp32 [N,H,W]
 * r3dp_sr_blend                out = a*alpha + b*(1-alpha), fp32 NCHW, alpha [N,1,H,W]
 * r3dp_sr_person_occlusion     out = clamp(torso_occlusion + (head_alpha > threshold ? 1 : head_alpha), 0, 1)
 * r3dp_sr_resize_aa_down2      F.interpolate(scale 1/2, bilinear, antialias=True): x [N,C,2h,2w] -> y [N,C,h,w] fp32 */
int r3dp_sr_tc_conv(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W, int ksize,
                    int act, void* y_f16, r3dp_stream_t stream);
/* large_sr (LargeSynthesisBlock0/1 + ResBlock2d, modules/eg3ds/models/superresolution.py:263-329):
 * r3dp_sr_tc_conv_res  r3dp_sr_tc_conv with act 3 = ReLU and an optional residual (NHWC fp16, the output's shape) added AFTER the activation:
 *                      ResBlock2d's `out = act(conv2(act(conv1(x)))) + x`
 * r3dp_sr_tc_torgb_ex  plain 1x1 conv to RGB; same_res != 0: img_out = img_prev[N,3,H,W] + conv1x1(x) + b  (`rgb = rgb + self.to_rgb(x)`) */
int r3dp_sr_tc_conv_res(const void* x_f16, const void* wp_f16, const float* bias, int N, int Nw, int I, int O, int H, int W, int ksize,
                        int act, const void* residual_f16, void* y_f16, r3dp_stream_t stream);
int r3dp_sr_tc_torgb_ex(const void* x_f16, const float* wrgb, const float* brgb, const float* img_prev, int same_res, int N, int Nw, int C,
                        int H, int W, float* img_out, r3dp_stream_t stream);
/* htbsr_head_weight_fuse_mode v1 / v3 (sr_with_ref.py:96-104,126-152):
 * r3dp_sr_alpha_mix   out[...,0:C] = xa * alpha + xb * (1 - alpha), fp16 NHWC with pixel strides stride_a / stride_b (v1's feature blend)
 * r3dp_sr_alpha_gate  out [N,1,H,W] fp32 = min(sigmoid(logit), cap): logit = channel 0 of an NHWC fp16 tensor (+ channel lo_off when lo_off > 0: split
 *                     output of r3dp_sr_tcx_conv) = tail of head_torso_alpha_predictor + the cap by the head weights (v3) */
int r3dp_sr_alpha_mix(const void* xa_f16, int stride_a, const void* xb_f16, int stride_b, const float* alpha, int C, int N, int H, int W,
                      void* out_f16, r3dp_stream_t stream);
int r3dp_sr_alpha_gate(const void* logits_f16, int stride, int lo_off, const float* cap, int N, int H, int W, float* out, r3dp_stream_t stream);
int r3dp_sr_tc_layer_torgb_noup(const void* x_f16, const void* wp_f16, const float* bias, const float* wrgb, const float* brgb,
                                const float* img_prev, int N, int Nw, int I, int O, int H, int W, void* y_f16, float* img_out,
                                r3dp_stream_t stream);
int r3dp_sr_alpha_cat(const void* xa_f16, int Ca, int stride_a, const void* xb_f16, int Cb, int stride_b, const float* alpha, int N,
                      int H, int W, void* out_f16, r3dp_stream_t stream);
/* xb_shared != 0: xb holds ONE frame [1,H,W,Cb] read by every frame of the batch (per-clip constant features, e.g. bg_encoder(ref_bg)). */
int r3dp_sr_alpha_cat_ex(const void* xa_f16, int Ca, int stride_a, const void* xb_f16, int Cb, int stride_b, int xb_shared, const float* alpha,
                         int N, int H, int W, void* out_f16, r3dp_stream_t stream);
int r3dp_sr_blend(const float* a, const float* b, const float* alpha, int N, int C, int H, int W, float* out, r3dp_stream_t stream);
int r3dp_sr_person_occlusion(const float* head_alpha, const float* torso_occlusion, float threshold, int N, int H, int W, float* out,
                             r3dp_stream_t stream);
int r3dp_sr_resize_aa_down2(const float* x, int N, int C, int h_out, int w_out, float* y, r3dp_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* R3DP_B200_H */
