/* libvfi_b200.so - C ABI of the B200-native frame-interpolation hot path (RIFE 4.6 first).
 *
 * The reference (Fannovel16/ComfyUI-Frame-Interpolation @ 26545cc) has no native library: its "FFI" is
 * (a) PyTorch ATen calls from vfi_models/rife/rife_arch.py and (b) cupy RawModule launches that pass
 * `(int32 n, raw device pointers...)` on torch's current stream (vfi_models/ops/cupy_ops/softsplat.py:206-224).
 * This header is what a maintainer binds instead (ctypes stub in INTEGRATION.md).  Conventions:
 *   - plain pointers and sizes only, no torch types; device pointers are owned by the caller (PyTorch);
 *   - every function returns 0 on success or a negative VFI_E_* code; vfi_last_error() gives the text
 *     (thread-local);  the Python host raises RuntimeError, mirroring the reference's exception behaviour;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream); no hidden synchronisation
 *     unless the function name says *_host or *_sync;
 *   - images are float32 NHWC in [0,1] exactly as ComfyUI's IMAGE type (rife/__init__.py:146,239).
 */
#ifndef VFI_B200_H
#define VFI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VFI_OK 0
#define VFI_E_INVALID (-1)   /* bad argument / unsupported configuration */
#define VFI_E_CUDA (-2)      /* CUDA runtime or kernel error */
#define VFI_E_STATE (-3)     /* e.g. forward before weights were loaded */
#define VFI_E_NOTIMPL (-4)

#define VFI_OPERAND_F16 0    /* conv operands fp16, fp32 accumulate (node dtype float32 / float16) */
#define VFI_OPERAND_BF16 1   /* conv operands bf16, fp32 accumulate (node dtype bfloat16) */

#define VFI_RIFE46_NUM_TENSORS 120   /* IFNet("4.6").state_dict() - rife_arch.py:404-408 */
#define VFI_RIFE47_NUM_TENSORS 124   /* IFNet("4.7"): + encode.{0,1}.{weight,bias} - rife_arch.py:409-417 */
#define VFI_RIFE417_NUM_TENSORS 128  /* + encode.cnn0..cnn3 weight, bias (Head_417, rife_arch.py:356-363) */
#define VFI_RIFE426_NUM_TENSORS 158  /* IFNet("4.26"): 5 blocks x 30 + Head cnn0..cnn3 weight, bias (rife_arch.py:453-459) */
#define VFI_MAX_BATCH 16

typedef struct vfi_ctx vfi_ctx;

/* library / context ------------------------------------------------------------------------------------ */
const char* vfi_last_error(void);
const char* vfi_version(void);
/* Creates a context bound to CUDA device `device` (its own compute/copy streams, workspace, weights). */
int vfi_create(int device, vfi_ctx** out);
int vfi_destroy(vfi_ctx* ctx);
/* Number of kernels this library has launched through `ctx` since creation (bench.py "gpu_launches"). */
int64_t vfi_launch_count(const vfi_ctx* ctx);
/* Pairs interpolated per internal pass (1..VFI_MAX_BATCH, default 8); replaces the node's batch_size knob
 * (rife/__init__.py:64-69) - it changes scheduling only, never results. */
int vfi_set_batch(vfi_ctx* ctx, int batch);

/* Replaces: IFNet(arch_ver="4.6").load_state_dict(torch.load(path)) - rife/__init__.py:129-133.
 * `tensors[i]` are HOST float32 arrays in state_dict order (block{b}.conv0.0.0.weight, .bias, conv0.1.0.weight,
 * .bias, 8 x convblock.{j}.{beta, conv.weight, conv.bias}, lastconv.0.weight, .bias; b = 0..3); `numel[i]` is
 * checked against the architecture.  Weights are repacked to the tensor-core operand layout on the device. */
int vfi_rife46_load(vfi_ctx* ctx, const float* const* tensors, const int64_t* numel, int n_tensors, int operand_type);
/* Same for any built arch: 46 (rife46.pth), 47 (rife47.pth / rife49.pth), 417 (rife417.pth) or 426 (rife426.pth: five
 * blocks, scale list [16,8,4,2,1]/scale_factor, rife/__init__.py:156-158; CKPT_NAME_VER_DICT rife/__init__.py:10-14;
 * state_dict order = blocks 0..3 then encode.0.weight, encode.0.bias, encode.1.weight, encode.1.bias).  The
 * vfi_rife46_forward / _interpolate_host entry points below run whichever arch was loaded. */
int vfi_rife_load(vfi_ctx* ctx, int arch, const float* const* tensors, const int64_t* numel, int n_tensors,
                  int operand_type);

/* Replaces: the body of the hot loop of RIFE_VFI.vfi - rife/__init__.py:185-207 - i.e.
 *   IFNet.forward(frame[f0[i]], frame[f1[i]], t[i], scale_list=[8,4,2,1]/scale_factor).clamp(0,1)
 * for n_tasks (pair, timestep) tasks.  DEVICE pointers:
 *   frames : [n_frames, H, W, C] float32 NHWC, C >= 3 (only the first 3 channels are read, vfi_utils.py:139)
 *   out    : [n_tasks, H, W, 3] float32 NHWC
 * scale_factor: the node's widget (rife/__init__.py:49, :156-160), one of 0.25, 0.5, 1, 2, 4 (with 2 / 4 the last one / two
 * blocks run on an up-scaled input).
 * Asynchronous on `stream`. */
int vfi_rife46_forward(vfi_ctx* ctx, const float* frames, int n_frames, int H, int W, int C, const int32_t* f0,
                       const int32_t* f1, const float* t, int n_tasks, float scale_factor, float* out, void* stream);

/* Replaces: the whole per-batch loop incl. `.to(device)` / `.cpu()` - rife/__init__.py:185-222 - with a
 * pipelined H2D / compute / D2H schedule.  HOST pointers (pinned memory gives full PCIe rate; pageable works):
 *   frames : [n_frames, H, W, C] float32;  out : frames of [H, W, 3] float32.
 * Task i is written to out + out_slot[i]*H*W*3 (out_slot == NULL: slot i), so the caller can have the
 * interpolated frames land directly between the pass-through frames of the node's output tensor
 * (rife/__init__.py:225-238) without a second host copy.
 * Only frames in [frame_lo, frame_hi) are uploaded (the shard of this rank); tasks must reference only those.
 * frame_slot (NULL or [n_frames]): source frame f in [frame_lo, frame_hi) with frame_slot[f] >= 0 is also copied unchanged
 * (first 3 channels) to out + frame_slot[f]*H*W*3 - the pass-through frames of rife/__init__.py:227-231 - by the library's
 * copy threads; with a page-locked `out` that copy doubles as the staging copy of the upload.
 * Pageable `frames` / `out` go through pinned staging rings (VFI_STAGE_MB, VFI_COPY_THREADS); the prepared-frame window
 * on the device is a ring of ~2 x batch + 1 frames whatever the clip length.
 * Synchronous: returns when `out` is complete. */
int vfi_rife46_interpolate_host(vfi_ctx* ctx, const float* frames, int n_frames, int H, int W, int C, int frame_lo,
                                int frame_hi, const int32_t* f0, const int32_t* f1, const float* t,
                                const int32_t* out_slot, const int32_t* frame_slot, int n_tasks, float scale_factor,
                                float* out);

/* Host utility for the node's output assembly (rife/__init__.py:225-238: every source frame is passed through between
 * the interpolated ones): frame i (first 3 of C channels) -> out + slot[i]*H*W*3 for every i with slot[i] >= 0, split over
 * `threads` host threads.  HOST pointers, any host memory; no GPU involved.  Runs beside vfi_rife46_interpolate_host. */
int vfi_host_copy_frames(const float* frames, int n_frames, int H, int W, int C, const int32_t* slot, float* out, int threads);

/* Primitive: backward bilinear warp == rife_arch.warp (rife_arch.py:31-70) ==
 * grid_sample(bilinear, padding_mode="border", align_corners=True) on a pixel-unit flow.  DEVICE pointers, NHWC:
 * img [B,H,W,C] float32, flow [B,H,W,2] float32 (x, y displacement in pixels), out [B,H,W,C]. */
int vfi_warp_bilinear_border(vfi_ctx* ctx, const float* img, const float* flow, float* out, int B, int H, int W, int C,
                             void* stream);

/* Op-level surface of vfi_models/ops (the names the reference's models import, vfi_models/ops/__init__.py:19-21).
 * DEVICE pointers, contiguous NCHW float32 exactly like the reference's cupy launches (cupy_ops/softsplat.py:206-224).
 *   vfi_softsplat_sum : softsplat_out (cupy_ops/softsplat.py:140-192): out[N,C,H,W] (zeroed here) += forward splat of in
 *                       along flow [N,2,H,W]; the avg/linear/soft modes are host-side arithmetic around it (:382-435)
 *   vfi_costvol_l1    : costvol_out (cupy_ops/costvol.py:4-43): out[N,81,H,W] = mean_c |one - two(+-4 shifted)|
 *   vfi_corr_dot      : kernel_Correlation_updateOutput (cupy_ops/correlation.py:31-99): out[N,81,H,W], zero padded
 *   vfi_sepconv       : sepconv_out (cupy_ops/sepconv.py:86-117): in [N,C,H+Kv-1,W+Kh-1], ver [N,Kv,H,W], hor [N,Kh,H,W] */
int vfi_softsplat_sum(vfi_ctx* ctx, const float* in, const float* flow, float* out, int N, int C, int H, int W,
                      void* stream);
/* Fused form of the wrapper modes of softsplat() (cupy_ops/softsplat.py:382-435): mode 0 avg, 1 linear, 2 soft (weight 1,
 * metric, exp(metric) per source pixel), eps 0 addeps (default) / 1 zeroeps / 2 clipeps; `norm` is a caller-provided
 * [N,1,H,W] scratch plane (the splatted weights); out [N,C,H,W] = splat(in * weight) / f(norm).  metric may be NULL for avg.
 * The splat and the channel-last volume form use scratch owned by the context; calls on different streams are ordered
 * against each other on it (the later call's stream waits for the earlier call), so one context may serve several streams. */
int vfi_softsplat_weighted(vfi_ctx* ctx, const float* in, const float* flow, const float* metric, int mode, int eps, float* out,
                           float* norm, int N, int C, int H, int W, void* stream);
int vfi_costvol_l1(vfi_ctx* ctx, const float* one, const float* two, float* out, int N, int C, int H, int W,
                   void* stream);
int vfi_corr_dot(vfi_ctx* ctx, const float* first, const float* second, float* out, int N, int C, int H, int W,
                 void* stream);
int vfi_sepconv(vfi_ctx* ctx, const float* in, const float* ver, const float* hor, float* out, int N, int C, int H,
                int W, int Kv, int Kh, void* stream);
/*   vfi_adacof        : kernel_AdaCoF_updateOutput (cupy_ops/adacof.py:5-62, wrapper :259-330): in [N,C,Hin,Win], weight /
 *                       offset_i / offset_j [N,F*F,Ho,Wo] with Hin = Ho + (F-1)*dilation, out [N,C,Ho,Wo]
 *   vfi_edt_pass      : kernel_dt (cupy_ops/batch_edt.py:9-41): one row pass of the separable squared distance transform,
 *                       data / out [bs,h,w]; batch_edt (:46-117) runs it twice around a transpose */
int vfi_adacof(vfi_ctx* ctx, const float* in, const float* weight, const float* offset_i, const float* offset_j, float* out,
               int N, int C, int Hin, int Win, int F, int dilation, int Ho, int Wo, void* stream);
int vfi_edt_pass(vfi_ctx* ctx, const float* data, float* out, int bs, int h, int w, float diam2, void* stream);

/* FILM (film_net) - SURVEY.md section 8 row a10 --------------------------------------------------------- */
#define VFI_FILM_NUM_TENSORS 82      /* film_arch.Interpolator().state_dict() (film_arch.py:377-393) */
/* Replaces: torch.jit.load(film_net_fp32.pt) - film/__init__.py:74.  `tensors[i]` are HOST float32 arrays in the
 * order of Interpolator.state_dict() (extract.extract_sublevels.convs.{0..3}.{0,1}.0.{weight,bias}, predict_flow.
 * _predictor._convs.{0..3}.0 / .4, predict_flow._predictors.{0,1,2}._convs..., fuse.output_conv, fuse.convs.{0..3}.
 * {0, 1.0, 2.0}); sizes are checked.  Weights are repacked to the streamed tensor-core operand layout. */
int vfi_film_load(vfi_ctx* ctx, const float* const* tensors, const int64_t* numel, int n_tensors, int operand_type);
/* Replaces: `model(x0, x1, dt)` in film/__init__.py:35-38 (Interpolator.forward, film_arch.py:458-459; the network
 * always predicts the midpoint, `dt` is not an input) for n_pairs independent pairs, optionally followed by the
 * node's clamp(0, 1) (:38).  DEVICE pointers: frames [n_frames, H, W, C] float32 NHWC (C >= 3, first three channels
 * read, vfi_utils.py:139), out [n_pairs, H, W, 3] float32 NHWC; f0 / f1: HOST index arrays.  H, W >= 64 (seven
 * pyramid levels), any other size as in the reference.  Asynchronous on `stream`. */
int vfi_film_forward(vfi_ctx* ctx, const float* frames, int n_frames, int H, int W, int C, const int32_t* f0,
                     const int32_t* f1, int n_pairs, int clamp01, float* out, void* stream);
/* Test / profiling hooks: route every FILM conv through the CUDA-core checker (1) or the tcgen05 kernel (0); run one
 * conv layer (group 0 = extract: layer 2*j + {0,1}; 1 = flow estimators: 4*predictor + conv; 2 = fusion: 3*k + conv)
 * on caller tensors (16-bit NHWC channel slices: pointer + pixel pitch in elements); static plan of a layer; tensor-core
 * MACs (unpadded channels) of the last forward. */
int vfi_film_debug_set_ref(vfi_ctx* ctx, int use_ref);
int vfi_film_debug_conv(vfi_ctx* ctx, int group, int layer, const void* src0, int pitch0, const void* src1, int pitch1,
                        void* out, int out_pitch, int B, int H, int W, int impl, void* stream);
int vfi_film_layer_plan(vfi_ctx* ctx, int group, int layer, int* c0, int* c1, int* n_total, int* ksize, int* n_cta,
                        int* nsplit, int* mt, int* a_slots, int* b_slots, int* smem_bytes);
int64_t vfi_film_last_macs(const vfi_ctx* ctx);
/* Host-only: vfi_film_load's weight packer on caller data (layout 0 = reference channel order padded to 64; layout 1 = a
 * fusion level's [wfeat0 C | wfeat1 C | misc 64] + nf decoder channels); `out` receives the packed 16-bit operand:
 * [split][k-block][tap][n_cta][64 ch, 16-byte chunks XOR (row & 7)]. */
int vfi_film_debug_pack_host(int layout, int C, int nf, int ksize, int n_total, int operand_type, const float* w,
                             int cout, int cin, uint16_t* out, int64_t out_cap, int* c0, int* c1, int* n_cta,
                             int* nsplit);

/* Sepconv (`Sepconv VFI` node) - SURVEY.md section 8 row a12 -------------------------------------------- */
#define VFI_SEPCONV_NUM_TENSORS 88   /* sepconv_enhanced.Network().state_dict() (sepconv_enhanced.py:536-598) */
/* Replaces: Network().load_state_dict(torch.load(path)) - sepconv/__init__.py:42-45.  HOST float32 arrays in
 * state_dict order (netInput, netEncode.0.netVer.{1..4}, netDecode.0.netHor.{0..3}, netDecode.0.netVer.{1..3}, netVerone,
 * netVertwo, netHorone, netHortwo); sizes are checked. */
int vfi_sepconv_load(vfi_ctx* ctx, const float* const* tensors, const int64_t* numel, int n_tensors, int operand_type);
/* Replaces: `model(frame_0, frame_1)` = Network.forward (sepconv_enhanced.py:605-706) for n_pairs independent pairs.
 * DEVICE pointers: frames [n_frames, H, W, C >= 3] float32 NHWC, out [n_pairs, H, W, 3] float32 NHWC (not clamped, like
 * the reference); f0 / f1: HOST index arrays.  Any H, W >= 2.  Asynchronous on `stream`. */
int vfi_sepconv_forward(vfi_ctx* ctx, const float* frames, int n_frames, int H, int W, int C, const int32_t* f0,
                        const int32_t* f1, int n_pairs, float* out, void* stream);
/* Test hooks: every conv through the CUDA-core checker (1) / the tcgen05 kernel (0); the host-only weight packer of
 * vfi_sepconv_load (a 3x3 conv packed as a stride-1 layer, or as the 2x2 conv over the space-to-depth input that runs
 * its stride-2 form). */
int vfi_sepconv_debug_set_ref(vfi_ctx* ctx, int use_ref);
int vfi_sepconv_debug_pack_host(int stride2, int cin, int cout, int n_total, int operand_type, const float* w, uint16_t* out,
                                int64_t out_cap, int* c0, int* n_cta, int* nsplit);

/* Test / profiling hooks (used by tests/ and bench.py only) --------------------------------------------- */
/* Run ONE convolution layer of block `block` (0..3; arch 4.26: 0..4): layer 0 = conv0.0, 1 = conv0.1, 2..9 = ResConv
 * 0..7, 10 = lastconv (flow + mask), 11 = arch 4.26 blocks 0..3: the 8 feature channels of lastconv, written as
 * [B, 4H, 4W, 8] 16-bit.  `in`/`out` are device tensors in the kernel-native layouts documented in DESIGN.md
 * (16-bit NHWC; layers 0/1 read space-to-depth inputs; layer 10 writes float4 flow + float mask planes).
 * impl 0 = tcgen05 kernel, 1 = CUDA-core checker with the same packed weights. */
int vfi_rife46_debug_layer(vfi_ctx* ctx, int block, int layer, const void* in, void* out, void* out_mask, int B, int H,
                           int W, int impl, void* stream);
/* Copies the full-resolution flow (float4 [batch,Hp,Wp]) and mask (float [batch,Hp,Wp]) of the LAST internal
 * pass into caller-provided DEVICE buffers (either may be NULL to only query Hp/Wp); synchronises. */
int vfi_rife46_debug_state(vfi_ctx* ctx, float* flow4_out, float* mask_out, int batch, int* Hp, int* Wp);
/* Static plan of a layer for (block, layer): shared-memory stages, CTA output channels, splits, smem bytes. */
int vfi_rife46_layer_plan(vfi_ctx* ctx, int block, int layer, int* stages, int* n_cta, int* nsplit, int* smem_bytes,
                          int64_t* macs_per_cell);
int vfi_sync(vfi_ctx* ctx);

/* Measurement hook (bench.py's roofline lines): while enabled, every internal pass of the RIFE forward schedule records
 * CUDA events on its launching stream around each kernel group - id = 10 * block + {0 front (warps + resample + concat,
 * rife_arch.py:238-249, :703-704), 1 conv0.0, 2 conv0.1, 3 the eight ResConvs, 4 lastconv}, 90 = the final warp / blend /
 * crop kernel (rife_arch.py:713-732).  vfi_rife_profile_read synchronises and returns, per group id, the summed device
 * time in ms and the number of spans; at most `cap` groups.  No counterpart in the reference (it has no timing code). */
int vfi_rife_profile(vfi_ctx* ctx, int enable);
int vfi_rife_profile_read(vfi_ctx* ctx, int32_t* ids, float* total_ms, int32_t* count, int cap, int* n_groups);

/* ---------------------------------------------------------------------------------------------------------------------
 * GMFSS Fortuna (union) building blocks - csrc/gmops.cu; the schedule that strings them together is host code
 * (comfyui-frame-interpolation_b200/gmfss.py), mirroring vfi_models/gmfss_fortuna/GMFSS_Fortuna_union_arch.py :1726-1857.
 * They replace what that file runs through ATen / cuDNN / cuBLAS between its softsplat calls: F.conv2d / conv_transpose2d
 * with the nn.PReLU in front and the residual adds behind (:1420-1688, :165-312), F.instance_norm (:165-215), nn.Linear /
 * torch.matmul / softmax / LayerNorm / GELU of the swin transformer (:315-685) and of the flow propagation (:688-803),
 * split_feature / merge_splits with torch.roll (:366-436, :1059-1131), PositionEmbeddingSine (:1015-1056),
 * local_correlation_softmax (:846-913), upsample_flow (:1220-1260), grid_sample / F.interpolate (:955-991, :1375-1417),
 * MetricNet's input assembly with the forward-backward check (:994-1013, :1429-1455), F.pixel_shuffle, torch.cat / slicing.
 * DEVICE pointers, contiguous float32, NCHW tensors (tokens: [B, L, C]); `stream` is the caller's CUDA stream; 0 = OK.
 * Argument meaning is documented at each kernel in csrc/gmops.cu. */
int vfi_gm_conv2d(const float* in, const float* w, const float* bias, const float* res1, const float* res2, float* out, int N, int Cin, int H, int W, int Cout, int k, int stride, int pad, int in_ctot, int in_coff, int out_ctot, int out_coff, int has_pre, float pre_slope, int post, float post_slope, void* stream);
int vfi_gm_conv2d_packed(const float* in, const float* wt, const float* bias, const float* res1, const float* res2, float* out, int N, int Cin, int H, int W, int Cout, int CoutP, int k, int stride, int pad, int in_ctot, int in_coff, int out_ctot, int out_coff, int has_pre, float pre_slope, int post, float post_slope, void* stream);
int vfi_gm_transpose(const float* src, float* dst, int nb, int R, int C, void* stream);
int vfi_gm_convt4(const float* in, const float* w, const float* bias, float* out, int N, int Cin, int H, int W, int Cout, int has_pre, float pre_slope, void* stream);
int vfi_gm_instance_norm(const float* in, float* out, int planes, int HW, float eps, int relu, void* stream);
int vfi_gm_layer_norm(const float* x, const float* gamma, const float* beta, const float* src, float* out, int rows, int C, float eps, void* stream);
int vfi_gm_softmax_rows(float* x, int rows, int L, void* stream);
int vfi_gm_gemm(int bt, const float* A, const float* B, const float* bias, const float* mask, float* C, int nb, int M, int N, int K, int lda, int ldb, int ldc, long long sA, long long sB, long long sC, float alpha, int nmask, int act, void* stream);
int vfi_gm_window(const float* src, float* dst, int B, int H, int W, int C, int k, int sh, int sw, int to_windows, void* stream);
int vfi_gm_nchw_tokens(const float* src, float* dst, int B, int C, int HW, int to_tokens, void* stream);
int vfi_gm_add_position(float* x, int B, int C, int H, int W, int k, void* stream);
int vfi_gm_local_match(const float* f0, const float* f1, float* flow, int B, int C, int H, int W, int R, void* stream);
int vfi_gm_local_prop(const float* q, const float* k, const float* flow, float* out, int B, int C, int H, int W, void* stream);
int vfi_gm_convex_up(const float* mask, const float* flow, float* up, int B, int H, int W, int f, void* stream);
int vfi_gm_warp_zeros(const float* in, const float* flow, float* out, int B, int C, int H, int W, void* stream);
int vfi_gm_resize(const float* in, float* out, int BC, int H, int W, int Ho, int Wo, int align, float mul, void* stream);
int vfi_gm_metric_input(const float* img0, const float* img1, const float* f01, const float* f10, float* out, int B, int H, int W, void* stream);
int vfi_gm_pixel_shuffle2(const float* in, float* out, int B, int C, int H, int W, void* stream);
int vfi_gm_axpby(const float* a, const float* b, float* out, long long n, float alpha, float beta, float gamma, int post, void* stream);
int vfi_gm_copy_slice(const float* src, float* dst, int B, int C, int Hs, int Ws, int Hd, int Wd, int s_ctot, int s_coff, int d_ctot, int d_coff, int src_nhwc, int dst_nhwc, const float* mean, const float* stdv, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VFI_B200_H */
