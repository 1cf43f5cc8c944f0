/*
 * md2_loss.h - C ABI of the B200-native view-synthesis loss path of monodepth2.
 *
 * The reference (GenkiK/monodepth2) is pure Python and has no FFI; the boundary a
 * maintainer would bind is the Python API of layers.py plus the two Trainer methods
 * that drive it.  Every entry point below names the reference interface it replaces
 * (file:line under /root/reference).  All pointers are CUDA *device* pointers to
 * contiguous fp32 NCHW tensors unless stated otherwise; `stream` is a cudaStream_t
 * passed as void*.  No torch types cross this boundary.  Every function returns
 * MD2_OK (0) or a negative md2_status; md2_status_string() names it.  All work is
 * enqueued asynchronously on `stream`; nothing synchronises the device.
 *
 * The shared library is libmd2loss.so (built by monodepth2_b200/build.py for sm_100a).
 */
#ifndef MD2_LOSS_H_
#define MD2_LOSS_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MD2_MAX_SCALES 4
#define MD2_MAX_SRC 4

typedef enum md2_status {
  MD2_OK = 0,
  MD2_ERR_INVALID_ARGUMENT = -1,
  MD2_ERR_UNSUPPORTED = -2,
  MD2_ERR_WORKSPACE_TOO_SMALL = -3,
  MD2_ERR_CUDA = -4
} md2_status;

/* Shape and flags of one loss evaluation: the subset of options.py that changes the
 * path (options.py:52-119) plus two tuning knobs. */
typedef struct md2_problem {
  int batch;                  /* opt.batch_size                        options.py:87  */
  int height, width;          /* opt.height / opt.width                options.py:52  */
  int num_scales;             /* len(opt.scales); levels: scale_level  options.py:64  */
  int num_src;                /* len(opt.frame_ids) - 1 (incl. "s")    options.py:80  */
  int automask;               /* !opt.disable_automasking              options.py:111 */
  int avg_reprojection;       /* opt.avg_reprojection                  options.py:108 */
  int align_corners;          /* grid_sample align_corners; the reference leaves it
                                 unspecified = 0 on torch>=1.3       trainer.py:384 */
  float min_depth, max_depth; /* opt.min_depth / opt.max_depth         options.py:69  */
  float disparity_smoothness; /* opt.disparity_smoothness              options.py:60  */
  int want_grad;              /* 0: forward only (Trainer.val under no_grad, trainer.py:330) */
  int rows_per_segment;       /* tuning: rows marched per warp job (0 = default) */
  int no_ssim;                /* opt.no_ssim: L1 only                  options.py:117 */
  int posecnn;                /* opt.pose_model_type == "posecnn" (options.py:101, trainer.py:366-375): T is built per
                                 scale from the pose leaves with the translation multiplied by the mean inverse depth
                                 of that scale; needs axisangle / translation for every source without a fixed T */
  int predictive_mask;        /* opt.predictive_mask (options.py:114, trainer.py:447-459); needs automask == 0 */
  int scale_level[MD2_MAX_SCALES]; /* opt.scales sorted ascending when it is not 0..n-1 (options.py:64, e.g. --scales 0 2;
                                 trainer.py:345,413 iterate the list, the dataloader always holds levels 0..3,
                                 trainer.py:127-135): scale slot s of every per-scale array below is pyramid level
                                 scale_level[s], (H >> level, W >> level), smoothness weight 1 / 2^level, and
                                 losses[1 + s] = losses["loss/<level>"].  All zero = levels 0..n-1 */
  /* ---- element type of the differentiable leaves (md2_dtype; all zero = every leaf fp32).  A bf16 / fp16 leaf is
   *      widened exactly to fp32 in workspace by one conversion launch at the start of the call, so every result is
   *      the fp32 call on the upcast leaves, bit for bit.  Losses, cam_T_cam, the side outputs and every grad_* output
   *      of md2_view_synthesis_loss stay fp32 (the Python wrapper rounds the gradients once to the leaf dtype). ---- */
  int disp_dtype;                   /* disp[s], every scale */
  int pose_dtype[MD2_MAX_SRC];      /* source f: T[f], or the axisangle[f] / translation[f] pair (a constant stereo_T
                                       may stay fp32 while the network's poses are bf16) */
  int pmask_dtype;                  /* pmask[s], every scale */
} md2_problem;

/* Element types of md2_problem's *_dtype fields and md2_scale_tensors_typed. */
typedef enum md2_dtype {
  MD2_DTYPE_F32 = 0,
  MD2_DTYPE_BF16 = 1,
  MD2_DTYPE_F16 = 2
} md2_dtype;

/* Tensors of one evaluation.  Names follow the reference's dict keys.  Per-scale arrays are indexed by scale SLOT
 * s = 0..num_scales-1; slot s is pyramid level md2_problem.scale_level[s] (= s for the default --scales 0 1 2 3), and
 * "H>>s" below reads H >> level. */
typedef struct md2_tensors {
  /* ---- inputs ---- */
  const float *target;                  /* inputs[("color",0,0)]         (B,3,H,W)      */
  const float *source[MD2_MAX_SRC];     /* inputs[("color",f,0)]         (B,3,H,W)      */
  const float *T[MD2_MAX_SRC];          /* outputs[("cam_T_cam",0,f)] or inputs["stereo_T"], (B,4,4) */
  int pose_requires_grad[MD2_MAX_SRC];  /* 0 for the constant stereo_T                   */
  const float *K;                       /* inputs[("K",0)]               (B,4,4)        */
  const float *inv_K;                   /* inputs[("inv_K",0)]           (B,4,4)        */
  const float *disp[MD2_MAX_SCALES];    /* outputs[("disp",s)]           (B,1,H>>s,W>>s) */
  const float *color[MD2_MAX_SCALES];   /* inputs[("color",0,s)]         (B,3,H>>s,W>>s) */
  const float *noise[MD2_MAX_SCALES];   /* tie-break draws of trainer.py:468-469, standard normal,
                                           (B,n_id,H,W), n_id = num_src | 1 (avg) ; NULL if !automask */
  /* ---- outputs ---- */
  float *losses;                        /* [0]=losses["loss"], [1+s]=losses["loss/s"]    */
  float *grad_disp[MD2_MAX_SCALES];     /* d loss / d disp_s             (B,1,H>>s,W>>s) */
  float *grad_T[MD2_MAX_SRC];           /* d loss / d cam_T_cam          (B,4,4); NULL allowed */
  /* ---- optional side outputs (NULL = skip), SURVEY.md 3.3 ---- */
  float *depth[MD2_MAX_SCALES];               /* outputs[("depth",0,s)]    (B,1,H,W)     */
  float *warped[MD2_MAX_SRC][MD2_MAX_SCALES]; /* outputs[("color",f,s)]    (B,3,H,W)     */
  float *identity_selection[MD2_MAX_SCALES];  /* outputs["identity_selection/s"] (B,H,W) */
  float *grad_depth_dbg[MD2_MAX_SCALES];      /* test hook: d loss / d upsampled disp_s (B,1,H,W) */
  /* ---- optional pose leaves (replaces layers.py:28-103 transformation_from_parameters as called from
   *      predict_poses, trainer.py:294-295): when axisangle[f] is non-NULL, T[f] is ignored and the call
   *      builds T_f = transformation_from_parameters(axisangle, translation, invert) itself; with want_grad the
   *      pose gradient is returned on the leaves.  3 floats per sample, pose_stride[f] floats between
   *      samples (6 for the [:, 0] view of PoseDecoder's (B,2,1,3) output, pose_decoder.py:49-54). ---- */
  const float *axisangle[MD2_MAX_SRC];
  const float *translation[MD2_MAX_SRC];
  int pose_stride[MD2_MAX_SRC];
  int pose_invert[MD2_MAX_SRC];               /* frame_id < 0                                  */
  float *cam_T_cam[MD2_MAX_SRC];              /* out: outputs[("cam_T_cam",0,f)] (B,4,4); NULL = internal scratch */
  float *grad_axisangle[MD2_MAX_SRC];         /* out (B,3) */
  float *grad_translation[MD2_MAX_SRC];       /* out (B,3) */
  /* ---- optional uint8 images (what MonoDataset holds before ToTensor, datasets/mono_dataset.py:106-109,
   *      156-185): when target_u8 is non-NULL the call reads the frames as bytes and converts them with
   *      x / 255 (bit-identical to torchvision's ToTensor) where it would have read the float images;
   *      target / source[] / color[] are then ignored and may be NULL.  Layout: u8_hwc != 0: (B,H,W,3)
   *      interleaved (numpy view of the PIL image), else (B,3,H,W) planar.  color_u8[0] may be NULL
   *      (= target_u8).  A quarter of the host-to-device bytes of the float entry. ---- */
  const unsigned char *target_u8;
  const unsigned char *source_u8[MD2_MAX_SRC];
  const unsigned char *color_u8[MD2_MAX_SCALES];
  int u8_hwc;
  /* ---- --predictive_mask (trainer.py:447-459): outputs["predictive_mask"][("disp", s)], (B,num_src,H>>s,W>>s)
   *      in (0,1); up-sampled to (H,W) inside the call, multiplied into the reprojection losses before the per-pixel
   *      minimum, and pushed towards 1 by 0.2 * BCE(mask, 1) added to loss/s.  grad_pmask[s] (same shape) receives
   *      d loss / d mask when want_grad; NULL = not wanted. ---- */
  const float *pmask[MD2_MAX_SCALES];
  float *grad_pmask[MD2_MAX_SCALES];
  /* ---- optional: a cudaEvent_t recorded (on any stream) after the last write of noise[]; the call waits for it
   *      right before the first kernel that reads the noise, not at its start, so the torch.randn draws of
   *      trainer.py:468-469 can run on another stream beside the identity pass.  NULL = noise[] is ready in
   *      stream order. ---- */
  void *noise_ready_event;
} md2_tensors;

int md2_version(void);
const char *md2_status_string(int status);

/* Bytes of device scratch the fused call needs for `p`.  fp32 copies of the reduced-precision leaves are reserved
 * only when a *_dtype field is non-zero; a dtype outside md2_dtype is MD2_ERR_INVALID_ARGUMENT. */
int md2_loss_workspace_bytes(const md2_problem *p, size_t *bytes);

/* Fused replacement for Trainer.generate_images_pred (trainer.py:341-391) followed by
 * Trainer.compute_losses (trainer.py:407-496) and, when want_grad, the adjoint that
 * losses["loss"].backward() (trainer.py:208) propagates to disp_s and cam_T_cam.
 * Threading: the library keeps one internal side stream and event pair per device (the small smoothness
 * kernels overlap the identity pass on it; fork/join by events, so the caller's stream order and CUDA-graph
 * capture of `stream` are preserved).  The enqueue of a call runs under a library lock, so calls may be issued from
 * several host threads (their side-stream work is then ordered one call after the other; the work on the callers'
 * streams is not).  `workspace` may be reused by successive calls on the same stream; two calls in flight on
 * different streams need two workspaces. */
int md2_view_synthesis_loss(const md2_problem *p, const md2_tensors *t,
                            void *workspace, size_t workspace_bytes, void *stream);

/* Measurement hook (bench.py roofline leg): when enabled, every md2_view_synthesis_loss call
 * records CUDA events on its stream around the dominant kernel (md2_march_roles);
 * md2_profile_march_ms waits for the last call's pair and returns its duration. */
int md2_profile_enable(int on);
int md2_profile_march_ms(float *ms);

/* ---- per-layer entry points: one per layers.py symbol on the path ---- */

/* layers.py:16-25 disp_to_depth -> scaled_disp, depth (either output may be NULL). n elements. */
int md2_disp_to_depth(const float *disp, float min_depth, float max_depth,
                      float *scaled_disp, float *depth, long long n, void *stream);
int md2_disp_to_depth_backward(const float *disp, float min_depth, float max_depth,
                               const float *grad_scaled, const float *grad_depth,
                               float *grad_disp, long long n, void *stream);

/* layers.py:139-168 BackprojectDepth.forward: depth (B,1,H,W), inv_K (B,4,4) -> (B,4,H*W). */
int md2_backproject_depth(const float *depth, const float *inv_K, float *cam_points,
                          int batch, int height, int width, void *stream);
int md2_backproject_depth_backward(const float *grad_cam_points, const float *inv_K,
                                   float *grad_depth, int batch, int height, int width, void *stream);

/* layers.py:171-193 Project3D.forward: points (B,4,H*W), K, T (B,4,4) -> grid (B,H,W,2). */
int md2_project3d(const float *points, const float *K, const float *T, float eps, float *pix_coords,
                  int batch, int height, int width, void *stream);
/* grad_points (B,4,H*W) and grad_T (B,4,4, accumulated from zero) may each be NULL. */
int md2_project3d_backward(const float *grad_pix, const float *points, const float *K, const float *T,
                           float eps, float *grad_points, float *grad_T,
                           int batch, int height, int width, void *stream);

/* trainer.py:384-387 F.grid_sample(img, grid, padding_mode="border"), bilinear. */
int md2_grid_sample_border(const float *img, const float *grid, float *out, int batch, int channels,
                           int in_h, int in_w, int out_h, int out_w, int align_corners, void *stream);
int md2_grid_sample_border_backward(const float *grad_out, const float *img, const float *grid,
                                    float *grad_grid, int batch, int channels, int in_h, int in_w,
                                    int out_h, int out_w, int align_corners, void *stream);

/* layers.py:218-248 SSIM.forward(x, y) -> clamp((1-SSIM)/2,0,1), (B,C,H,W). */
int md2_ssim(const float *x, const float *y, float *out, int batch, int channels, int height,
             int width, void *stream);
/* grad_x and grad_y may each be NULL. */
int md2_ssim_backward(const float *grad_out, const float *x, const float *y, float *grad_x,
                      float *grad_y, int batch, int channels, int height, int width, void *stream);

/* layers.py:202-215 get_smooth_loss(disp, img) -> scalar (loss[0]); scratch: 2 doubles. */
int md2_smooth_loss(const float *disp, const float *img, float *loss, void *scratch16,
                    int batch, int channels, int height, int width, void *stream);
int md2_smooth_loss_backward(const float *grad_loss, const float *disp, const float *img,
                             float *grad_disp, int batch, int channels, int height, int width,
                             void *stream);

/* layers.py:28-103 transformation_from_parameters(axisangle, translation, invert):
 * axisangle, translation (B,3) -> T (B,4,4); backward maps grad_T to the two leaves. */
int md2_pose_to_matrix(const float *axisangle, const float *translation, int invert, float *T,
                       int batch, void *stream);
int md2_pose_to_matrix_backward(const float *grad_T, const float *axisangle, const float *translation,
                                int invert, float *grad_axisangle, float *grad_translation,
                                int batch, void *stream);

/* ---- decoder tail feeding the path (SURVEY.md 8f-4): outputs[("disp", s)] = sigmoid(Conv3x3(C -> 1)(x)),
 * networks/depth_decoder.py:60-63 with Conv3x3 = ReflectionPad2d(1) + Conv2d(C, 1, 3), layers.py:119-136.
 * x (B,C,H,W), weight (1,C,3,3), bias (1) -> disp (B,1,H,W); pad + conv + bias + sigmoid in one pass. ---- */
int md2_dispconv_sigmoid(const float *x, const float *weight, const float *bias, float *disp,
                         int batch, int channels, int height, int width, void *stream);
/* grad_x (B,C,H,W), grad_weight (1,C,3,3) and grad_bias (1) are written (not accumulated); grad_x and
 * grad_weight may each be NULL (grad_bias is produced with grad_weight). */
int md2_dispconv_sigmoid_backward(const float *grad_disp, const float *disp, const float *x, const float *weight,
                                  float *grad_x, float *grad_weight, float *grad_bias,
                                  int batch, int channels, int height, int width, void *stream);
/* The same head on a bf16 / fp16 feature map (`dtype`, md2_dtype; MD2_DTYPE_F32 selects the fp32 kernels above):
 * x, disp, grad_disp and grad_x are in `dtype`; weight, bias, grad_weight and grad_bias are fp32.  x is read at 2 bytes
 * a value and widened exactly; the arithmetic is the fp32 kernels' (weights read in fp32 as stored, not rounded to
 * bf16 as autocast's conv2d does); disp and grad_x are the fp32 results rounded once to nearest-even. */
int md2_dispconv_sigmoid_typed(const void *x, const float *weight, const float *bias, void *disp, int dtype,
                               int batch, int channels, int height, int width, void *stream);
int md2_dispconv_sigmoid_backward_typed(const void *grad_disp, const void *disp, const void *x, const float *weight,
                                        void *grad_x, float *grad_weight, float *grad_bias, int dtype,
                                        int batch, int channels, int height, int width, void *stream);

/* ---- decoder stages (SURVEY.md 8f-4): the input of every ConvBlock of DepthDecoder.forward,
 * networks/depth_decoder.py:48-65 - upsample (layers.py:196-199), torch.cat and the ReflectionPad2d(1) of Conv3x3
 * (layers.py:106-136) - in one pass:
 *   out = ReflectionPad2d(1)(cat([nearest_up(x, up), skip], dim=1))
 * x (B,Cx,h,w); skip (B,Cs,up*h,up*w), or NULL with Cs = 0; out (B,Cx+Cs,up*h+2,up*w+2).  `height` and `width` are
 * x's.  up = 2 with a skip is the ("upconv", i, 1) input, up = 2 without one stage 0's, up = 1 without one the plain pad
 * of ("upconv", i, 0) and of a Conv3x3 ("dispconv", s) head.  x, skip, out and the gradients share `dtype` (md2_dtype).
 * up must be 1 or 2, up*h and up*w at least 2, Cx >= 1, Cs >= 0; out must have fewer than 2^31 elements
 * (else MD2_ERR_UNSUPPORTED).  Forward is pure data movement, bit-identical to torch's chain in every dtype. ---- */
int md2_upcat_pad(const void *x, const void *skip, void *out, int dtype, int batch, int x_channels,
                  int skip_channels, int height, int width, int up, void *stream);
/* The adjoint in gather form, without atomics (bitwise reproducible): each element of grad_x / grad_skip sums the
 * padded positions that read it - its own first, then the reflected ones - and grad_x sums its up x up children in
 * row-major order (ATen's upsample_nearest2d_backward), all in fp32 from 0.0f, rounded once to `dtype`.  grad_x and
 * grad_skip are written (not accumulated) and may each be NULL. */
int md2_upcat_pad_backward(const void *grad_out, void *grad_x, void *grad_skip, int dtype, int batch, int x_channels,
                           int skip_channels, int height, int width, int up, void *stream);

/* ---- monitoring path (SURVEY.md 8f-5): Trainer.compute_depth_losses, trainer.py:498-526, with
 * compute_depth_errors, layers.py:251-269.  depth = outputs[("depth",0,0)] (B,1,H,W), depth_gt (B,1,Hg,Wg);
 * metrics[7] = abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3 (device floats, the order of depth_metric_names,
 * trainer.py:105-106) over the pixels with gt > 0 inside crop [y0,y1) x [x0,x1) (153:371, 44:1197 in the reference),
 * after median scaling (torch.median = lower median, found exactly by radix select).  No host synchronisation. ---- */
int md2_depth_metrics_scratch_bytes(int batch, int gt_height, int gt_width, size_t *bytes);
int md2_depth_metrics(const float *depth, const float *depth_gt, float *metrics, void *scratch, size_t scratch_bytes,
                      int batch, int height, int width, int gt_height, int gt_width,
                      int crop_y0, int crop_y1, int crop_x0, int crop_x1, void *stream);

/* autograd glue (trainer.py:208, losses["loss"].backward()): dst[i] = src[i] * (*scale) for n_tensors <=
 * MD2_MAX_SCALE_TENSORS device tensors in one launch; `src`, `dst`, `numel` are HOST arrays, `scale` a device scalar. */
#define MD2_MAX_SCALE_TENSORS 16
int md2_scale_tensors(int n_tensors, const float *const *src, float *const *dst, const long long *numel,
                      const float *scale, void *stream);
/* The same with a destination element type per tensor (dst_dtype[i], md2_dtype; HOST array): dst[i] is the fp32
 * product src[i] * (*scale) rounded once to nearest-even (an overflow gives +-inf, never a saturated value), so a loss
 * scale applied before the rounding keeps fp16 gradients that the unscaled product would flush to zero.
 * Bitwise md2_scale_tensors for an fp32 destination.  One launch. */
int md2_scale_tensors_typed(int n_tensors, const float *const *src, void *const *dst, const int *dst_dtype,
                            const long long *numel, const float *scale, void *stream);

/* ---- colour pyramid on the GPU (SURVEY.md 8f-3): replaces the per-frame host work of
 * MonoDataset.preprocess, datasets/mono_dataset.py:57,82-86,98-103 - torchvision Resize with
 * Image.ANTIALIAS on PIL images = PIL.Image.resize(size, LANCZOS), scale i built from scale i-1.
 * Byte-exact with Pillow's 8-bit fixed-point resample (Resample.c); coefficient tables are computed on the host
 * and uploaded when the plan is created (synchronous; do it once, outside CUDA-graph capture). ---- */
typedef struct md2_resize_plan md2_resize_plan;
int md2_resize_plan_create(int in_h, int in_w, int out_h, int out_w, md2_resize_plan **plan);
void md2_resize_plan_destroy(md2_resize_plan *plan);
/* bytes of device scratch one call needs (the uint8 temporary of the horizontal pass) */
int md2_resize_scratch_bytes(const md2_resize_plan *plan, int batch, size_t *bytes);
/* in: (B,in_h,in_w,3) when hwc != 0, else (B,3,in_h,in_w); out: same layout at (out_h,out_w). */
int md2_resize_lanczos_u8(const md2_resize_plan *plan, const unsigned char *in, unsigned char *out,
                          void *scratch, size_t scratch_bytes, int batch, int hwc, void *stream);

/* ---- colour augmentation on the GPU (SURVEY.md 8f-3): replaces `self.to_tensor(color_aug(f))` of
 * MonoDataset.preprocess with color_aug = transforms.ColorJitter.get_params(brightness, contrast, saturation, hue)
 * (datasets/mono_dataset.py:60-70,107-109,169-176): torchvision's adjust_brightness / contrast / saturation / hue
 * on uint8 RGB images, i.e. Pillow's Image.blend against black / the mean gray level / the "L" image and the
 * RGB -> HSV -> RGB round trip with the hue byte shifted - byte-exact with Pillow.  One parameter set per image
 * (`params`: DEVICE array of n_images entries; the reference draws one set per dataset item and applies it to every
 * frame and scale of the item).  order[k]: 0 brightness, 1 contrast, 2 saturation, 3 hue, -1 skip, applied for
 * k = 0..3 (ColorJitter.get_params' fn_idx); hue_shift = uint8(int32(hue_factor * 255)).
 * in / out: (n,H,W,3) when hwc != 0, else (n,3,H,W); scratch: n_images * 8 bytes. ---- */
typedef struct md2_color_jitter {
  int order[4];
  float brightness, contrast, saturation;
  int hue_shift;
} md2_color_jitter;
int md2_color_jitter_u8(const unsigned char *in, unsigned char *out, const md2_color_jitter *params, void *scratch,
                        size_t scratch_bytes, int n_images, int height, int width, int hwc, void *stream);

/* ---- the training batch of MonoDataset.__getitem__ + preprocess on the GPU (SURVEY.md 8f-3,
 * datasets/mono_dataset.py:90-109,136-185, kitti_dataset.py get_color): from the native uint8 frames a worker loaded,
 * the flip, the LANCZOS pyramid and the per-scale colour augmentation of every (sample, frame) image of a batch, in
 * 2 * num_scales + 3 launches whatever the batch size, frame count and mix of native sizes.
 *
 * Image n of a batch is described by a job.  Its native frame is (height, width, 3) uint8 HWC (np.array of the PIL
 * image) at byte `offset` of `frames`; `flip` mirrors it horizontally before the resize (get_color's
 * transpose(FLIP_LEFT_RIGHT)); `sample` is its row of `params` (one md2_color_jitter per dataset item, shared by its
 * frames and scales; a row whose order is all -1 is the identity); `size` is the index
 * md2_batch_plan_add_native_size returned for (height, width).
 *
 * Outputs hold every level back to back: level s (h_s = height >> s, w_s = width >> s) starts at element
 * n_images * 3 * sum_{t<s} h_t * w_t, image n of it at n * 3 * h_s * w_s, NCHW.
 *   out_color:     ("color", f, s): the resized bytes, uint8, or float32 x / 255 (= ToTensor) when color_f32 != 0;
 *   out_color_aug: ("color_aug", f, s): float32 ToTensor of the jittered level (the jitter runs after each resize, with
 *                  the level's own contrast mean, as the reference's preprocess does).
 * Creating the plan and adding a size are synchronous (tables are built on the host in double arithmetic, as Pillow
 * does, and uploaded); md2_batch_build_u8 only enqueues, so once every native size is added it can be captured in a
 * CUDA graph.  `jobs` is read on the host for validation, `jobs_dev` (the same records on the device) by the kernels. */
#define MD2_BATCH_MAX_SIZES 64
typedef struct md2_batch_job {
  long long offset;           /* byte offset of the native frame in `frames` */
  int height, width;          /* native size */
  int size;                   /* index of (height, width) in the plan */
  int flip;                   /* non-zero: mirrored (do_flip) */
  int sample;                 /* row of `params` */
  int reserved;
} md2_batch_job;
typedef struct md2_batch_plan md2_batch_plan;
int md2_batch_plan_create(int height, int width, int num_scales, md2_batch_plan **plan);
void md2_batch_plan_destroy(md2_batch_plan *plan);
/* index of (h, w) among the plan's native sizes; tables are built and uploaded the first time a size is added */
int md2_batch_plan_add_native_size(md2_batch_plan *plan, int h, int w, int *index);
/* bytes of device scratch one md2_batch_build_u8 call over n_images needs */
int md2_batch_scratch_bytes(const md2_batch_plan *plan, int n_images, int color_f32, size_t *bytes);
int md2_batch_build_u8(const md2_batch_plan *plan, const unsigned char *frames, size_t frames_bytes,
                       const md2_batch_job *jobs, const md2_batch_job *jobs_dev, int n_images,
                       const md2_color_jitter *params, int n_samples, void *out_color, int color_f32,
                       float *out_color_aug, void *scratch, size_t scratch_bytes, void *stream);

/* ---- KITTI raw depth_gt on the GPU (SURVEY.md 8f-3): KITTIRAWDataset.get_depth (datasets/kitti_dataset.py) =
 * generate_depth_map (kitti_utils.py) + skimage.transform.resize(order=0, preserve_range=True, mode='constant')
 * to (out_h, out_w) + np.fliplr when flipped, then the float32 rounding of MonoDataset.__getitem__.
 *
 * Job n is one sample.  Its scan is the velodyne file as read: n_points x 4 float32 (x, y, z, reflectance; the 4th
 * column is ignored) at byte `offset` of `scans`, 16-byte aligned.  P is P_velo2im (row-major 3x4, float64) and
 * (height, width) the native image size im_shape, both from the drive's calibration (host code, cached per camera).
 * Per point, in float64: (u', v', w) = P (x, y, z, 1), col = rint(u'/w) - 1, row = rint(v'/w) - 1; points with x >= 0
 * landing inside the native image store w (x when vel_depth != 0); the last point at a pixel wins, then each group of
 * the reference's sub2ind (a pixel, plus (r+1, 0) for (r, W-1)) holding more than one point gets the group's minimum
 * at the pixel of its first point; negatives become 0.  The order-0 resize takes output o from native index
 * floor((o + 0.5) * (n / n_out) - 0.5 + 0.5) (float64, in that order).  out: (n_jobs, 1, out_h, out_w) float32.
 * An output size equal to the native size gives generate_depth_map itself (export_gt_depth.py's use).
 *
 * Every native axis must be shorter than 1.25 x the output axis (beyond that skimage's anti-aliasing filter smooths
 * the map) and the native width at least 2: else MD2_ERR_UNSUPPORTED.  `jobs` is read on the host for validation,
 * `jobs_dev` (the same records on the device) by the kernels.  The scratch size depends only on n_jobs and the output
 * size, and md2_velo_depth only enqueues (3 launches), so one allocation and one captured CUDA graph serve every batch
 * of that shape.  Bitwise reproducible.
 * The maps are the reference's bit for bit with one exception: a zero is always +0.0.  The reference keeps a -0.0 stored
 * value (only a velodyne x of -0.0 under vel_depth gives one) through some of numpy's reductions and clips and not
 * others, so its sign there depends on numpy's summation order. ---- */
typedef struct md2_velo_job {
  double P[12];               /* P_velo2im, row-major 3x4 */
  long long offset;           /* byte offset of the scan in `scans` */
  int n_points;               /* rows of the scan */
  int height, width;          /* native image size (im_shape) */
  int flip;                   /* non-zero: np.fliplr after the resize (do_flip) */
  int vel_depth;              /* non-zero: store the velodyne x instead of the camera depth */
  int reserved;
} md2_velo_job;
int md2_velo_depth_scratch_bytes(int n_jobs, int out_h, int out_w, size_t *bytes);
int md2_velo_depth(const unsigned char *scans, size_t scans_bytes, const md2_velo_job *jobs,
                   const md2_velo_job *jobs_dev, int n_jobs, float *out, int out_h, int out_w, void *scratch,
                   size_t scratch_bytes, void *stream);

/* ---- baseline JPEG decoding on the GPU: the frames of kitti_dataset.py get_color, pil_loader's
 * Image.open(f).convert("RGB"), byte for byte what Pillow's libjpeg-turbo gives, for SOF0 8-bit Huffman-coded
 * three-component YCbCr streams with luma sampling 1x1, 2x1 or 2x2 and chroma 1x1, any restart interval.
 *
 * The host (monodepth2_b200/jpeg.py) walks the markers, removes the 0xFF00 stuffing and the RSTn markers, and lays
 * out per image, inside `data`: the entropy-coded segments (one per restart interval), each starting on a
 * MD2_JPEG_CHUNK_BYTES boundary of the image's entropy area and zero-padded to the next; the segment table
 * (n_segments md2_jpeg_segment); and an md2_jpeg_tables record (several images may share one).
 * Chunks are numbered across the call: image n owns chunks [chunk_offset, chunk_offset + n_chunks), and blocks
 * [block_offset, block_offset + mcus * blocks per MCU) of the coefficient scratch; both offsets are the running sums
 * over the images before it.  The image is written as (height, width, 3) uint8 HWC at byte out_offset of `frames`.
 *
 * status (device, n_images uint32) gets per image the MD2_JPEG_* bits below; 0 is a clean decode.  A stream that sets
 * one may leave any bytes in its frame, but the call never reads or writes outside its buffers.
 * The scratch size depends only on n_images and the capacity (max_chunks, max_blocks); md2_jpeg_decode only enqueues
 * (a memset and four kernels), so one allocation and one captured CUDA graph serve every batch within the capacity.
 * `jobs` is read on the host for validation, `jobs_dev` (the same records on the device) by the kernels. ---- */
#define MD2_JPEG_CHUNK_BYTES 64
#define MD2_JPEG_BAD_CODE 1u          /* a Huffman code no table holds */
#define MD2_JPEG_EXHAUSTED 2u         /* a segment's data ended before its last MCU */
#define MD2_JPEG_BAD_INDEX 4u         /* a run took the coefficient index past 63 */
#define MD2_JPEG_BAD_SEGMENT 8u       /* a segment record outside the image's chunks */
typedef struct md2_jpeg_huff {        /* jpeg_make_d_derived_tbl */
  unsigned short look[256];           /* (code length << 8) | symbol for codes of <= 8 bits, else 0 */
  int maxcode[18];                    /* largest code of each length, -1 if none; maxcode[17] = 0xFFFFF */
  int valoffset[18];                  /* huffval index = code + valoffset[length] */
  unsigned char huffval[256];
} md2_jpeg_huff;
typedef struct md2_jpeg_tables {
  md2_jpeg_huff dc[2], ac[2];
  unsigned short quant[4][64];        /* natural (row-major) order */
} md2_jpeg_tables;
typedef struct md2_jpeg_segment {
  int chunk;                          /* first chunk, counted from the image's first */
  int bytes;                          /* unstuffed entropy bytes */
} md2_jpeg_segment;
typedef struct md2_jpeg_job {
  long long out_offset;               /* byte offset of the decoded frame in `frames` */
  long long entropy_offset;           /* byte offset of the image's entropy area (its chunk 0) in `data` */
  long long segments_offset;          /* byte offset of the segment table in `data`, 8-byte aligned */
  long long tables_offset;            /* byte offset of the md2_jpeg_tables record in `data`, 8-byte aligned */
  long long block_offset;             /* first block in the coefficient scratch */
  int chunk_offset, n_chunks;         /* the image's chunks */
  int n_segments;                     /* ceil(mcus / restart_interval), 1 without restart interval */
  int restart_interval;               /* MCUs per segment, 0: one segment */
  int height, width;
  int h_samp, v_samp;                 /* luma sampling: (1, 1), (2, 1) or (2, 2) */
  int dc_table[3], ac_table[3];       /* 0 or 1 per component (Y, Cb, Cr) */
  int quant_table[3];                 /* 0..3 per component */
  int reserved;
} md2_jpeg_job;
int md2_jpeg_decode_scratch_bytes(int n_images, long long max_chunks, long long max_blocks, size_t *bytes);
int md2_jpeg_decode(const unsigned char *data, size_t data_bytes, const md2_jpeg_job *jobs, const md2_jpeg_job *jobs_dev,
                    int n_images, unsigned char *frames, size_t frames_bytes, unsigned int *status,
                    long long max_chunks, long long max_blocks, void *scratch, size_t scratch_bytes, void *stream);

/* ---- PNG decoding on the GPU: the frames of kitti_dataset.py get_color for KITTI's own .png files, pil_loader's
 * Image.open(f).convert("RGB"), byte for byte what Pillow gives, for 8-bit truecolour non-interlaced PNGs.
 *
 * The host (monodepth2_b200/png.py) checks the chunks and the 2-byte zlib header and lays out per image, inside
 * `data`, the concatenated IDAT payloads from the first byte after the zlib header: the deflate data, and after it
 * whatever the file holds (the Adler-32 trailer, or nothing, or more).  Images are numbered across the call by two
 * running sums: stream_index over stream_bytes and raw_offset over the inflated size height * (3 * width + 1).  The
 * image is written as (height, width, 3) uint8 HWC at byte out_offset of `frames`.
 *
 * The Adler-32 trailer is read where zlib reads it, from the byte after the final block, and checked when all four
 * bytes are present and the inflated data is complete there or shorter (zlib's stream end).  A stream that ends a
 * positive whole number of rows short with a good trailer gives the image with zero rows after it, as Pillow does;
 * any other early end is MD2_PNG_EXHAUSTED.  One case differs from Pillow: Pillow feeds zlib one IDAT piece (at most
 * 64 KB) at a time and skips the check of a complete image's trailer when the trailer is not in the piece that
 * completes the last row; here it is always checked.  status (device, n_images
 * uint32) gets per image the MD2_PNG_* bits below; 0 is a clean decode.  A stream that sets one may leave any bytes
 * in its frame, but the call never reads or writes outside its buffers.  The scratch size depends only on n_images
 * and the capacity (max_stream_bytes, max_raw_bytes); md2_png_decode only enqueues (a memset and six kernels), so
 * one allocation and one captured CUDA graph serve every batch within the capacity.  `jobs` is read on the host for
 * validation, `jobs_dev` (the same records on the device) by the kernels. ---- */
#define MD2_PNG_BAD_CODE 1u           /* an invalid block type, code set, code, repeat or stored length */
#define MD2_PNG_DISTANCE 2u           /* a distance back past the start of the data */
#define MD2_PNG_EXHAUSTED 4u          /* the data ended before the last row (truncated, or too little output) */
#define MD2_PNG_BAD_FILTER 8u         /* a row's filter type above 4 */
#define MD2_PNG_CHECKSUM 16u          /* the Adler-32 trailer differs from the inflated data's */
#define MD2_PNG_CAPACITY 32u          /* the image lies outside the buffers or the capacity (a replayed CUDA graph
                                         fed a larger batch): skipped */
#define MD2_PNG_MAX_SIDE 16384
typedef struct md2_png_job {
  long long out_offset;               /* byte offset of the decoded frame in `frames` */
  long long stream_offset;            /* byte offset of the stream in `data`, 4-byte aligned; data holds it rounded up
                                         to whole 4-byte words */
  long long stream_index;             /* running sum of stream_bytes over the images before */
  long long raw_offset;               /* running sum of height * (3 * width + 1) over the images before */
  int stream_bytes;
  int height, width;                  /* 1..MD2_PNG_MAX_SIDE */
  int reserved;
} md2_png_job;
int md2_png_decode_scratch_bytes(int n_images, long long max_stream_bytes, long long max_raw_bytes, size_t *bytes);
int md2_png_decode(const unsigned char *data, size_t data_bytes, const md2_png_job *jobs, const md2_png_job *jobs_dev,
                   int n_images, unsigned char *frames, size_t frames_bytes, unsigned int *status,
                   long long max_stream_bytes, long long max_raw_bytes, void *scratch, size_t scratch_bytes,
                   void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MD2_LOSS_H_ */
