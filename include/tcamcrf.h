/*
 * tcamcrf.h -- C ABI of libtcamcrf.so: the B200-native (sm_100a) DenseCRF-loss
 * hot path of TCAM (permutohedral-lattice bilateral filter, loss, gradient,
 * temporal-CAM max and fg/bg seeding).
 *
 * Two groups of entry points:
 *
 *  1. DROP-IN (host pointers).  Same names, argument order and meaning as the
 *     functions the reference exposes to Python through SWIG:
 *       bilateralfilter / bilateralfilter_batch
 *           <- dlib/crf/crfwrapper/bilateralfilter/bilateralfilter.hpp:10-12
 *              (SWIG typemaps bilateralfilter.i:21-25)
 *       colorbilateralfilter / colorbilateralfilter_batch
 *           <- dlib/crf/crfwrapper/colorbilateralfilter/colorbilateralfilter.hpp:10-16
 *     They copy host->device, run the CUDA path on the current device and copy
 *     the result back (pipelined in chunks of frames).  The reference functions
 *     return void; these return a status code (0 = ok) as the only extension.
 *
 *  2. DEVICE API (device pointers, stream-ordered, capture-safe: no hidden
 *     synchronisation, no allocation).  This is what the python modules
 *     DenseCRFLoss / ColorDenseCRFLoss / TCAMSeeder call.  The caller owns
 *     every buffer, including the workspace.
 *
 * Layouts are the reference's: images planar [N,C,H,W] float32 holding 0..255,
 * segmentations / outputs planar [N,K,H,W] float32.
 *
 * Errors never exit(): every function returns a TCAMCRF_* status and
 * tcamcrf_last_error() describes the last failure of the calling thread.
 * Conditions that are only detectable on the device (hash table or vertex
 * pool overflow, lattice coordinate out of the packed-key range) are recorded
 * in the workspace status word: the outputs of that call are then filled with
 * NaN -- never silently wrong -- and tcamcrf_workspace_status() reports why.
 */
#ifndef TCAMCRF_H_
#define TCAMCRF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TCAMCRF_VERSION 104

/* host-side status codes */
#define TCAMCRF_OK 0
#define TCAMCRF_ERR_INVALID 1   /* bad argument (null pointer, non-positive size, unsupported dim) */
#define TCAMCRF_ERR_WORKSPACE 2 /* workspace too small or misaligned */
#define TCAMCRF_ERR_CUDA 3      /* a CUDA runtime call or kernel launch failed */
#define TCAMCRF_ERR_NO_DEVICE 4 /* no sm_100 device visible */
#define TCAMCRF_ERR_DEVICE_STATUS 5 /* device-side condition, see TCAMCRF_DEV_* */

/* device-side status bits (workspace status word) */
#define TCAMCRF_DEV_TABLE_FULL 1  /* a frame's hash table overflowed */
#define TCAMCRF_DEV_POOL_FULL 2   /* vertex pool overflowed */
#define TCAMCRF_DEV_KEY_RANGE 4   /* lattice coordinate outside the packed-key range */

/* element types of logits (the *_typed entry points) */
#define TCAMCRF_DTYPE_F32 0  /* float32 */
#define TCAMCRF_DTYPE_F16 1  /* IEEE half */
#define TCAMCRF_DTYPE_BF16 2 /* bfloat16 */

/* feature kinds */
#define TCAMCRF_FEAT_XY_RGB 0 /* (x/sxy, y/sxy, c0/srgb, ..): d = 2 + channels; reference bilateralfilter: channels = 3 */
#define TCAMCRF_FEAT_COLOR 1  /* (c0/srgb, ..): d = channels; reference colorbilateralfilter */

typedef struct tcamcrf_config {
    int feat;          /* TCAMCRF_FEAT_* */
    int channels;      /* image planes used as features (DIM of the colour filter) */
    int image_stride_planes; /* planes between consecutive images in `images`; the reference's
                                batch functions hard-code 3 (bilateralfilter.cpp:51, colorbilateralfilter.cpp:50) */
    float sigma_rgb;
    float sigma_xy;    /* ignored for TCAMCRF_FEAT_COLOR */
    float hash_load;   /* load factor the primary table tier would have at 1.2 vertices per pixel; 0 -> default (0.25).
                          Larger lattices spill into a worst-case-sized overflow tier, so any value is safe. */
    float pool_factor; /* vertex pool size as a fraction of the worst case (d+1)*H*W per frame; 0 -> 1.0 */
    int chunk_frames;  /* frames processed per pass (bounds the workspace); 0 -> default: 64, fewer for large frames
                          (workspace kept within ~16 GiB).  Always lowered when 32-bit vertex / entry indices need it. */
    float loss_weight; /* the module's `weight` (dense_crf_loss.py:118-122) folded into the loss kernels:
                          loss_dev[0] = loss_weight * (-sum(segs*AS)/n_norm), two separately rounded operations like
                          the reference's `self.weight * Function.apply(...)`; 0 -> 1 (the plain loss) */
} tcamcrf_config;

int tcamcrf_version(void);
const char *tcamcrf_last_error(void);

/* Number of sm_100 devices the library can run on (0 -> every compute call fails). */
int tcamcrf_device_count(void);

/* Bytes of device workspace the device API needs for this problem (0 on invalid arguments). */
size_t tcamcrf_workspace_bytes(const tcamcrf_config *cfg, int N, int K, int H, int W);

/* AS = alpha * Slice(Blur(Splat(segs))) per frame and class.
 * images_dev [N, stride_planes, H, W], segs_dev/as_dev [N,K,H,W]; all float32 on the current device.
 * Replaces the compute of bilateralfilter_batch / colorbilateralfilter_batch
 * (bilateralfilter.cpp:42-55, colorbilateralfilter.cpp:41-54). */
int tcamcrf_filter(const tcamcrf_config *cfg, const float *images_dev, const float *segs_dev, float *as_dev,
                   int N, int K, int H, int W, void *workspace, size_t workspace_bytes, void *cuda_stream);

/* Same as tcamcrf_filter, with 8-bit images (planar uint8, same plane layout): the loader-side
 * format SURVEY.md §8(f).1 asks for.  Features are float(u8)/sigma, i.e. identical values. */
int tcamcrf_filter_u8(const tcamcrf_config *cfg, const uint8_t *images_dev, const float *segs_dev, float *as_dev,
                      int N, int K, int H, int W, void *workspace, size_t workspace_bytes, void *cuda_stream);

/* A^T * segs: the same filter with the blur axes applied in the opposite order (d..0).  Each single-axis blur is
 * symmetric and slice is the transpose of splat, so this is exactly the transposed operator.  Not used by the
 * reference (its backward is -2*g*AS/N, dense_crf_loss.py:73, which treats A as symmetric); it backs the opt-in
 * exact gradient -(g/N)*(A + A^T)*segs of DenseCRFLoss(exact_gradient=True) (SURVEY.md §8f.4). */
int tcamcrf_filter_transposed(const tcamcrf_config *cfg, const void *images_dev, int images_u8, const float *segs_dev,
                               float *ats_dev, int N, int K, int H, int W, void *workspace, size_t workspace_bytes,
                               void *cuda_stream);

/* Host-side check of the packed-key range (no device work): 1 when frames whose image planes lie in
 * [0, max_value] cannot produce a lattice coordinate outside the 64-bit packed keys for this configuration
 * (sigma too small for the lattice dimension: the fields hold 20 bits per coordinate for d <= 3, 15 / 12 / 10 bits
 * for d = 4 / 5 / 6), else 0.  The device detects the same condition per call (TCAMCRF_DEV_KEY_RANGE, outputs NaN);
 * this lets a caller refuse a configuration up front with a clear message.  The reference's int16 keys wrap silently
 * instead (permutohedral.cpp:245-248). */
int tcamcrf_key_range_ok(const tcamcrf_config *cfg, int H, int W, float max_value);

/* Frames one pass works on for this problem (what tcamcrf_workspace_bytes sizes the workspace for): cfg->chunk_frames
 * or the default 64, capped by N and lowered for large frames (32-bit indices, ~16 GiB default workspace).  Also the
 * most frames one lattice of tcamcrf_lattice_build can hold.  0 on invalid arguments. */
int tcamcrf_chunk_frames(const tcamcrf_config *cfg, int N, int K, int H, int W);

/* Lattice reuse.  tcamcrf_lattice_build runs the image-only stages (tables, per-pixel vertices and weights, blur
 * links: Permutohedral::init, permutohedral.cpp:115-297) for N <= chunk_frames frames into `workspace`;
 * tcamcrf_lattice_apply then filters any number of [N,K,H,W] tensors through that lattice
 * (Permutohedral::compute, permutohedral.cpp:507-572): out = A*segs, or A^T*segs when `transposed` != 0; with
 * loss_dev != NULL also loss_dev[0] = -sum(segs*out)/n_norm.  The workspace (sized by tcamcrf_workspace_bytes for
 * the same cfg, N, K, H, W) IS the lattice: keep it untouched between the calls.  This is what the reference does
 * per image inside bilateralfilter() (one init, K computes, bilateralfilter.cpp:28-37), what the exact-gradient
 * backward needs (same lattice, transposed blur order) and what mean-field inference needs (one lattice, many
 * iterations: DenseCRFFilter, dlib/crf/crf_post_processing.py:99-128). */
int tcamcrf_lattice_build(const tcamcrf_config *cfg, const void *images_dev, int images_u8, int N, int K, int H,
                          int W, void *workspace, size_t workspace_bytes, void *cuda_stream);
int tcamcrf_lattice_apply(const tcamcrf_config *cfg, const float *segs_dev, float *out_dev, float *loss_dev, int N,
                          int K, int H, int W, float n_norm, int transposed, void *workspace, size_t workspace_bytes,
                          void *cuda_stream);

/* Forward of the DenseCRF loss: as_dev as above and loss_dev[0] = -sum(segs*AS)/n_norm
 * (dlib/crf/dense_crf_loss.py:56-66).  n_norm is the reference's N (the local batch size). */
int tcamcrf_loss_forward(const tcamcrf_config *cfg, const float *images_dev, const float *segs_dev, float *as_dev,
                         float *loss_dev, int N, int K, int H, int W, float n_norm, void *workspace,
                         size_t workspace_bytes, void *cuda_stream);
int tcamcrf_loss_forward_u8(const tcamcrf_config *cfg, const uint8_t *images_dev, const float *segs_dev,
                            float *as_dev, float *loss_dev, int N, int K, int H, int W, float n_norm,
                            void *workspace, size_t workspace_bytes, void *cuda_stream);

/* tcamcrf_loss_forward (loss_dev != NULL) / tcamcrf_filter (loss_dev == NULL) for frames that are still in HOST
 * memory -- what the reference's trainer passes: raw_img stays on the CPU (dlib/learning/train_wsol.py:1128) and
 * DenseCRFLossFunction.forward receives it every step (dlib/crf/dense_crf_loss.py:36-49).  images_host
 * [N, stride_planes, H, W] float32, or uint8 when images_u8 != 0 (a quarter of the bytes: SURVEY.md 8(f).1), pinned
 * for a truly asynchronous copy (pageable memory works, the driver then stages it), is copied into images_stage_dev (same size, device) section by section on a copy stream of the
 * library, and the lattice of every section is built on cuda_stream as soon as its frames are in: the copy hides
 * behind the lattice build instead of preceding it.  Stream-ordered (events only, no synchronisation): the call
 * returns once everything is queued, and images_host must stay untouched until cuda_stream has passed this call.
 * logits != 0: segs_dev holds logits (see tcamcrf_loss_forward_logits below). */
int tcamcrf_loss_forward_host_frames(const tcamcrf_config *cfg, const void *images_host, void *images_stage_dev,
                                     int images_u8, const float *segs_dev, float *as_dev, float *loss_dev, int logits,
                                     int N, int K, int H, int W, float n_norm, void *workspace,
                                     size_t workspace_bytes, void *cuda_stream);

/* Backward: grad_seg = ((-2 * grad_out[0]) * AS) / n_norm, the reference's expression and rounding
 * order (dlib/crf/dense_crf_loss.py:73).  count = N*K*H*W. */
int tcamcrf_loss_backward(const float *as_dev, const float *grad_out_dev, float *grad_seg_dev, size_t count,
                          float n_norm, void *cuda_stream);

/* The same with the module's weight folded in: grad_seg = ((-2 * (grad_out[0] * weight)) * AS) / n_norm -- what
 * autograd computes for `weight * loss` (the multiplication's backward hands grad_out * weight to
 * DenseCRFLossFunction.backward), without the two extra elementwise launches. */
int tcamcrf_loss_backward_weighted(const float *as_dev, const float *grad_out_dev, float *grad_seg_dev, size_t count,
                                   float n_norm, float weight, void *cuda_stream);

/* The same loss taken directly from LOGITS (SURVEY.md §8f.1): segs = softmax(logits) over the K classes is
 * formed on the fly inside the splat and slice kernels and never stored, and the backward pass goes through the
 * softmax in the same kernel:  dz_k = p_k * (g_k - sum_j p_j g_j),  g = ((-2*grad_out)*AS)/n_norm.
 * Replaces `F.softmax(fcams, dim=1)` + DenseCRFLoss in ConRanFieldTcams.forward (dlib/losses/tcam.py:109-115).
 * images_dev is float32 (images_u8 = 0) or uint8 (images_u8 = 1).  K >= 2. */
int tcamcrf_loss_forward_logits(const tcamcrf_config *cfg, const void *images_dev, int images_u8,
                                const float *logits_dev, float *as_dev, float *loss_dev, int N, int K, int H, int W,
                                float n_norm, void *workspace, size_t workspace_bytes, void *cuda_stream);
int tcamcrf_loss_backward_logits(const float *as_dev, const float *logits_dev, const float *grad_out_dev,
                                 float *grad_logits_dev, int N, int K, int H, int W, float n_norm, void *cuda_stream);
int tcamcrf_loss_backward_logits_weighted(const float *as_dev, const float *logits_dev, const float *grad_out_dev,
                                          float *grad_logits_dev, int N, int K, int H, int W, float n_norm,
                                          float weight, void *cuda_stream);

/* The logits entry points for logits of any TCAMCRF_DTYPE_* element type: what a model run under autocast hands
 * the loss (fp16 or bf16), read as they are, with no float32 copy.  Logits are widened on load (exact) and
 * everything after is the float32 computation: AS, the loss and the workspace stay float32, and the gradient is
 * written in the logits' type, rounded once from the float32 value.  Given the same AS, the gradient has the bits of
 * the float32 entry point on the widened logits followed by a cast to the logits' type.  Logits must be aligned to
 * their element size.  The float32 entry points above are these with TCAMCRF_DTYPE_F32.  An unknown dtype code
 * returns TCAMCRF_ERR_INVALID. */
int tcamcrf_loss_forward_logits_typed(const tcamcrf_config *cfg, const void *images_dev, int images_u8,
                                      const void *logits_dev, int logits_dtype, float *as_dev, float *loss_dev, int N,
                                      int K, int H, int W, float n_norm, void *workspace, size_t workspace_bytes,
                                      void *cuda_stream);
/* tcamcrf_loss_forward_host_frames with logits != 0, for logits of any TCAMCRF_DTYPE_* type. */
int tcamcrf_loss_forward_host_frames_typed(const tcamcrf_config *cfg, const void *images_host, void *images_stage_dev,
                                           int images_u8, const void *logits_dev, int logits_dtype, float *as_dev,
                                           float *loss_dev, int N, int K, int H, int W, float n_norm, void *workspace,
                                           size_t workspace_bytes, void *cuda_stream);
/* grad_logits_dev has the logits' element type. */
int tcamcrf_loss_backward_logits_typed(const float *as_dev, const void *logits_dev, int logits_dtype,
                                       const float *grad_out_dev, void *grad_logits_dev, int N, int K, int H, int W,
                                       float n_norm, float weight, void *cuda_stream);

/* Reads the device status word of a workspace (synchronises the stream).  Returns 0 or TCAMCRF_DEV_* bits
 * in *dev_status; also writes the number of lattice vertices of the last chunk to *vertices (may be NULL). */
int tcamcrf_workspace_status(void *workspace, void *cuda_stream, int *dev_status, int *vertices);

/* Lattice introspection for parity tests: builds the lattice of ONE image and copies out, to host memory,
 * per-(pixel,remainder) vertex ids [H*W*(d+1)] (pixel-major like the reference's offset_), barycentric
 * weights [H*W*(d+1)], the number of vertices, and the neighbour table [(d+1)*M*2] (when nbr_cap >= that).
 * Vertex ids are an arbitrary relabelling of the reference's. */
int tcamcrf_debug_lattice(const tcamcrf_config *cfg, const float *image_host, int H, int W, int32_t *offset_host,
                          float *bary_host, int *vertices, int32_t *nbr_host, size_t nbr_cap);

/* Seeding introspection for tests: the random words and Exp(1) draws tcam_seed_fused makes without q_dev, through
 * the same device functions.  tcam_debug_seed_draws: for every (b < B, side < 2, pixel < HW), the Philox4x32-10 word
 * of counter (pixel, 2b + side, 0x5eed, 0) keyed by the two words at rng_dev, and its draw; words_dev / draws_dev
 * [B,2,HW].  tcam_debug_exp_draws: the draw of each of the n words at words_dev. */
int tcam_debug_seed_draws(const unsigned int *rng_dev, int B, int HW, unsigned int *words_dev, float *draws_dev,
                          void *cuda_stream);
int tcam_debug_exp_draws(const unsigned int *words_dev, int n, float *draws_dev, void *cuda_stream);

/* ---- drop-in host API (reference names and argument lists) ---- */
int bilateralfilter(float *image, int len_image, float *in, int len_in, float *out, int len_out, int H, int W,
                    float sigmargb, float sigmaxy);
int bilateralfilter_batch(float *images, int len_images, float *ins, int len_ins, float *outs, int len_outs, int N,
                          int K, int H, int W, float sigmargb, float sigmaxy);
int colorbilateralfilter(float *image, int len_image, float *in, int len_in, float *out, int len_out, int H, int W,
                         float sigmargb, int DIM);
int colorbilateralfilter_batch(float *images, int len_images, float *ins, int len_ins, float *outs, int len_outs,
                               int N, int K, int H, int W, float sigmargb, int DIM);

/* Host-pointer fwd+bwd of the loss in one call (what bench.py's e2e leg times):
 * images/segs in host memory, writes loss_host[0], grad_host [N,K,H,W] (for grad_out = 1 * weight). */
int tcamcrf_loss_fwd_bwd_host(const tcamcrf_config *cfg, const float *images_host, const float *segs_host,
                              float *loss_host, float *grad_host, int N, int K, int H, int W, float grad_out);

/* Tuning knobs (sweeps and tests; never needed for correctness).  The library reads TCAMCRF_<NAME> from the
 * environment once, at first use; this sets a knob at run time instead.  name, with or without the TCAMCRF_ prefix:
 *   "DENSE"          1 / 0: the row-cooperative splat on / off, whatever the density hint says
 *   "BUILD_DEDUP"    1 / 0: the shared-memory dedup lattice build on / off, whatever the density hint says
 *   "HIMG_SECTIONS"  sections (1..64) of a chunk on the host-frames path (tcamcrf_loss_forward_host_frames)
 *   "HOST_GROUPS"    value-stage groups (1..64) per chunk on the host-pointer path (tcamcrf_loss_fwd_bwd_host)
 *   "HOST_SECTION0"  frames of the first lattice section on the host-pointer path
 *   "HOST_GROW"      factor by which each later section on the host-pointer path grows over the one before
 *   "HOST_TRACE"     1: print the timeline of every host-pointer call to stderr (runs the schedule eagerly)
 * value < 0 (or 0 where 0 is not meaningful) restores the default.  Any other name is refused. */
int tcamcrf_set_tuning(const char *name, int value);

/* ---- measurement hooks (bench.py) ----
 * Stage timing brackets every pipeline stage with CUDA events on the caller's stream (not capture-safe while
 * enabled).  Stages: 0 build, 1 neighbour, 2 splat, 3 blur (d+1 launches), 4 slice, 5 loss reduce/finish, 6 backward,
 * 7 prepare (table clear), 8 temporal max / seeding. */
#define TCAMCRF_STAGES 9
void tcamcrf_profile_enable(int on);
/* Waits for the recorded events; fills accumulated milliseconds and kernel launches per stage. */
int tcamcrf_profile_read(double *ms, long long *launches, int reset);
/* Kernels launched by this library since it was loaded (all threads). */
long long tcamcrf_launch_count(void);

/* ---- temporal CAM max + seeding (dlib/datasets/wsol_loader.py:585-600, dlib/cams/tcam_seeding.py:178-260) ---- */

/* out[b] = max_t cams[b,t] with torch.maximum's NaN propagation; cams_dev [B,T,HW], out_dev [B,HW]. */
int tcam_temporal_max(const float *cams_dev, float *out_dev, int B, int T, int HW, void *cuda_stream);

/* ROI by connected components, one thread block per sample: GetRoiSingleCam.__call__ with roi_method
 * 'roi_high_density' (largest_only = 0) or 'roi_largest' (1), dlib/cams/tcam_seeding.py:347-412.
 * cams_dev [B,H*W]; thresh_dev [B] on the 0..255 scale (tcam_otsu_roi's thresholds, or thresh*255);
 * roi_dev [B,H*W] int64 0/1: the selected 4-connected component of cam*255 >= thresh; bbox_dev [B,4] int32
 * x0,y0,x1,y1 (cv2.boundingRect convention of dlib/utils/wsol.py:133-137); bbox_mask_dev [B,H*W] float 0/1.
 * p_min_area: a densest component smaller than p_min_area*H*W gives way to the largest one; a double, so that the
 * product is the reference's float64 (h*w)*p_min_area_roi and a component of exactly that area is kept. */
size_t tcam_roi_components_scratch_bytes(int B, int H, int W);
int tcam_roi_components(const float *cams_dev, const float *thresh_dev, long long *roi_dev, float *bbox_mask_dev,
                        int *bbox_dev, int B, int H, int W, int largest_only, double p_min_area, void *scratch_dev,
                        size_t scratch_bytes, void *cuda_stream);

/* The same with the loader's per-frame re-normalisation first (re_normalize_cam, dlib/datasets/wsol_loader.py:
 * 594-595, 630-635): every frame becomes nan_to_num(exp((cam + 1e-6) * h) / max over the frame) before the max.
 * h <= 0 means no re-normalisation (sl_tc_knn_t == 0). */
int tcam_temporal_max_renorm(const float *cams_dev, float *out_dev, int B, int T, int HW, float h, void *cuda_stream);

/* Trainer.prepare_std_cams_disq (dlib/learning/train_wsol.py:417-432) in one pass: nan_to_num(nan=0, posinf=1,
 * neginf=0) -> bilinear resize to H x W (align_corners=False) -> nan_to_num.  cams_dev [B,h,w], out_dev [B,H,W]. */
int tcam_prepare_std_cams(const float *cams_dev, float *out_dev, int B, int h, int w, int H, int W, void *cuda_stream);

/* Temporal max fused with seed selection, for a whole batch in one launch (one thread block per sample and
 * per fg/bg).  Replaces, per sample, _SFG.forward / _SBG.forward (dlib/cams/tcam_seeding.py:498-592):
 *   value = max_t cams[b,t] (* roi) + 1e-8;  candidates = the n_cand largest (fg) / smallest (bg) values,
 *   ties broken by pixel index like torch's stable sort;  selected = top-k of p / q over the candidates in
 *   row-major order, p = value (weighted fg) or 1, q = the caller's Exp(1) draws (torch.multinomial without
 *   replacement is exactly this), so the result is bit-exact given the same draws.
 * cams_dev [B,T,HW]; roi_dev [B,HW] int64 or NULL (fg only); q_dev: draws of all (sample, fg|bg) pairs,
 * q_offset_dev [B,2] their starts; n_cand_dev [B,2] (0 = emit no seed); k_fg/k_bg seeds per sample.
 * Outputs: cam_max_dev [B,HW]; sel_dev [B,2,kmax] pixel indices (-1 = unused); scratch_dev [B,2,HW] floats. */
int tcam_seed_select(const float *cams_dev, int T, const int64_t *roi_dev, const float *q_dev,
                     const int *q_offset_dev, const int *n_cand_dev, int k_fg, int k_bg, int weighted_fg, int B, int HW,
                     float *cam_max_dev, float *scratch_dev, int *sel_dev, int kmax, void *cuda_stream);

/* Label map from the selected seeds: flat ksz x ksz dilation of fg and bg seeds, pixels claimed by both ->
 * ignore; out_dev [B,H,W] int64 in {ignore_idx, 0, 1} (dlib/cams/tcam_seeding.py:212-254). */
int tcam_seed_labels(const int *sel_dev, int kmax, int B, int H, int W, int ksz, long long ignore_idx,
                     int64_t *out_dev, void *cuda_stream);

/* The whole seeding step of a batch in ONE launch (a thread-block cluster of 8 blocks per sample): temporal max
 * (cam_max_dev [B,H*W] out), candidate counts, fg and bg selection, label map.  Replaces the per-sample loop of
 * TCAMSeeder.forward (dlib/cams/tcam_seeding.py:232-254) with _OneSample / _SFG / _SBG (:433-592) inside it:
 *   - candidate counts like the reference: none for a flat CAM (cam.min() == cam.max(), :465); fg: int(max_p * roi.sum())
 *     as a float32 product (:510,519), or n_fg_fixed = int(max_p*H*W) without a roi (:515); bg: n_bg = int(min_p*H*W)
 *     (:567).  n_cand_dev [B,2], when given, overrides them (a caller that sized its draws from its own counts);
 *   - candidates = the n largest (fg, on cam*roi + 1e-8) / smallest (bg, on cam + 1e-8) values, ties to the lowest
 *     pixel index (stable sort); selected = top-k of p / q, p = value (weighted_fg) or 1;
 *   - q: the caller's Exp(1) draws in row-major candidate order (q_dev + q_offset_dev [B,2]: bit-identical to
 *     tcam_seed_select, i.e. to the reference's multinomial given the same stream), or, with q_dev == NULL, drawn in
 *     the kernel by Philox4x32-10 keyed with the two words at rng_dev (fresh per call, e.g. from torch's generator):
 *     draw = -logf((2m + 1) * 2^-24), m = the top 23 bits of the word of (sample, side, pixel), so every draw is
 *     finite and > 0 (tcam_debug_seed_draws returns them);
 *   - labels_dev [B,H,W] int64 (or NULL): flat ksz x ksz dilation of the seeds, conflicts -> ignore (:239-254).
 * sel_dev [B,2,kmax] pixel indices (-1 = unused).  tcam_seed_fused_supported: the slice of a frame (H*W/8 pixels,
 * 8 bytes each) must fit the shared memory of an SM and kmax <= 32; otherwise use tcam_seed_select + tcam_seed_labels.
 * It answers for the current device: ask with the device current that tcam_seed_fused will run on. */
int tcam_seed_fused_supported(int HW, int kmax);
int tcam_seed_fused(const float *cams_dev, int T, const int64_t *roi_dev, const float *q_dev, const int *q_offset_dev,
                    const int *n_cand_dev, const unsigned int *rng_dev, float max_p, int n_fg_fixed, int n_bg, int k_fg,
                    int k_bg, int weighted_fg, int B, int H, int W, int ksz, long long ignore_idx, float *cam_max_dev,
                    int *sel_dev, int kmax, int64_t *labels_dev, void *cuda_stream);

/* Cross-entropy on the seeds without the label map: SelfLearningTcams (dlib/losses/tcam.py:48-77) =
 * CrossEntropyLoss(ignore_index)(fcams, seeds) with 'mean' over the labelled pixels, and the labelled pixels are the
 * ksz x ksz windows around the seeds in sel_dev [B,2,kmax] (side 0 = foreground -> class 1, side 1 = background ->
 * class 0; a pixel both sides reach is ignored, tcam_seeding.py:239-254).  Same value and gradient as torch's call
 * on tcam_seed_labels' map, from 2*kmax*ksz^2 work items per sample instead of four passes over [B,K,H,W].
 * forward: scratch_dev = 1 + 2*B floats, zero before the first call (left clean); loss_dev [1] (NaN when nothing is
 * labelled, like torch); count_dev [1] labelled pixels (kept for backward); optionally total_dev [1] = add_dev[0] +
 * weight * loss (add_dev: another loss term already computed on the stream, e.g. the CRF's; may be NULL).
 * backward: grad_logits_dev [B,K,H,W] += (grad_out * scale) * d loss / d logits  (in place, on top of whatever is there). */
int tcam_seed_ce_forward(const float *logits_dev, const int *sel_dev, int kmax, int B, int K, int H, int W, int ksz,
                         float *scratch_dev, float *loss_dev, float *count_dev, const float *add_dev, float weight,
                         float *total_dev, void *cuda_stream);
int tcam_seed_ce_backward(const float *logits_dev, const int *sel_dev, int kmax, int B, int K, int H, int W, int ksz,
                          const float *count_dev, const float *grad_out_dev, float scale, float *grad_logits_dev,
                          void *cuda_stream);

/* The same for logits of any TCAMCRF_DTYPE_* element type (see tcamcrf_loss_forward_logits_typed); the loss, count
 * and total stay float32.  The backward's grad_logits_dev has the logits' type: each labelled element becomes
 * round(widen(old) + (grad_out * scale) * d loss / d logits), one rounding. */
int tcam_seed_ce_forward_typed(const void *logits_dev, int logits_dtype, const int *sel_dev, int kmax, int B, int K,
                               int H, int W, int ksz, float *scratch_dev, float *loss_dev, float *count_dev,
                               const float *add_dev, float weight, float *total_dev, void *cuda_stream);
int tcam_seed_ce_backward_typed(const void *logits_dev, int logits_dtype, const int *sel_dev, int kmax, int B, int K,
                                int H, int W, int ksz, const float *count_dev, const float *grad_out_dev, float scale,
                                void *grad_logits_dev, void *cuda_stream);

/* Backward of crf_weight * CRF(softmax(logits)) + ce_weight * CE(logits, seeds) (the forward being
 * tcamcrf_loss_forward_logits_typed with loss_weight = crf_weight and tcam_seed_ce_forward_typed): writes
 * grad_logits_dev [B,K,H,W] (the logits' type) = tcamcrf_loss_backward_logits_typed(weight = crf_weight), with the
 * cross-entropy's gradient (scale = ce_weight) added on the labelled pixels.  Every element is rounded once from its
 * float32 value: the bits of the float32 sequence (CRF gradient, then tcam_seed_ce_backward in place) cast to the
 * logits' type. */
int tcam_crf_seed_ce_backward_typed(const float *as_dev, const void *logits_dev, int logits_dtype, const int *sel_dev,
                                    int kmax, int ksz, const float *count_dev, const float *grad_out_dev, int B, int K,
                                    int H, int W, float n_norm, float crf_weight, float ce_weight,
                                    void *grad_logits_dev, void *cuda_stream);

/* ROI of every CAM of a batch by Otsu's threshold: roi = (cam*255 >= otsu(floor(cam*255))), 1/0 as int64, the
 * 'roi_all' branch of GetRoiSingleCam (dlib/cams/tcam_seeding.py:316-345,419-430; scikit-image threshold_otsu
 * on a 256-bin np.histogram, float32 edges).  cams_dev [B,HW] float32, roi_dev [B,HW], thresh_dev [B] or NULL. */
int tcam_otsu_roi(const float *cams_dev, int64_t *roi_dev, float *thresh_dev, int B, int HW, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* TCAMCRF_H_ */
