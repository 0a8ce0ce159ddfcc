/*
 * idc_b200.h -- C ABI of the B200-native Local Hints Network forward
 * (interactive deep colorization hot path).
 *
 * The reference has NO native interface: its operator boundary for this path is the
 * Python call
 *     self.net.forward(img_l_mc, input_ab_mc, input_mask_mult, mask_cent)
 *         /root/reference/data/colorize_image.py:263   (ColorizeImageTorch.net_forward)
 *         /root/reference/data/colorize_image.py:308   (ColorizeImageTorchDist.net_forward)
 *     implemented by SIGGRAPHGenerator.forward
 *         /root/reference/models/pytorch/model.py:134-175
 * and, for the Caffe backend, the blob write + net.forward() at
 *         /root/reference/data/colorize_image.py:425-431, 452-463.
 * Every entry point below names the reference statement it replaces.  Plain pointers
 * and sizes only (no torch types); see INTEGRATION.md for the ctypes binding.
 *
 * Conventions
 *   - return value: 0 = IDC_OK, <0 = error (idc_last_error gives the text).
 *   - all image tensors are FP32, NCHW, contiguous (the reference's layout:
 *     model.py:139-141 builds [1,C,H,W] from numpy [C,H,W]).
 *   - idc_forward takes DEVICE pointers and is asynchronous on `stream`;
 *     idc_forward_host takes HOST pointers, copies through pinned staging buffers and
 *     returns after the results are in host memory.
 *   - a ctx is bound to one device, is not thread-safe, and owns packed weights +
 *     activation workspace.  Callers own all I/O buffers.
 *   - H and W must be multiples of 8 (three ::2 subsamplings + three x2 deconvs,
 *     model.py:149-151, :75,:86,:96).
 */
#ifndef IDC_B200_H_
#define IDC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct idc_ctx idc_ctx;

enum {
  IDC_OK = 0,
  IDC_ERR_ARG = -1,          /* bad argument / null pointer / bad shape            */
  IDC_ERR_CUDA = -2,         /* a CUDA call or kernel failed                        */
  IDC_ERR_STATE = -3,        /* wrong call order (e.g. forward before finalize)     */
  IDC_ERR_KEY = -4,          /* unknown / missing state_dict key                    */
  IDC_ERR_UNSUPPORTED = -5,  /* e.g. not an sm_100 device                           */
  IDC_ERR_WATCHDOG = -6      /* a device-side pipeline wait timed out               */
};

/* idc_create flags */
enum {
  IDC_FLAG_DIST = 1u << 0,        /* also run model_class + softmax (model.py:159-160)           */
  IDC_FLAG_ENGINE_SIMT = 1u << 1, /* FP32 CUDA-core engine (exact FP32, slow); default = tcgen05 */
  IDC_FLAG_FAST_FP16 = 1u << 2,   /* single-pass FP16 operands (1 MMA / product, ~6e-2 ab error);
                                     default = 2-term split FP16 (3 MMAs / product, <=1e-3)      */
  IDC_FLAG_GLOBAL_HINTS = 1u << 3,/* global-hints branch (models/global_model/deploy_nodist.prototxt:38-172,501-527) */
  IDC_FLAG_NO_GRAPH = 1u << 4,    /* do not capture the forward into a CUDA graph               */
  IDC_FLAG_KEEP_CONV10 = 1u << 5, /* materialise conv10_2 (debug); default fuses model_out into model10.1 */
  IDC_FLAG_CAFFE313 = 1u << 6     /* Caffe-spec 313-bin hyper-column head (deploy_nopred.prototxt:651-850) */
};

/* dtype codes for idc_load_tensor */
enum { IDC_F32 = 0, IDC_F64 = 1, IDC_I64 = 2 };

/* Library / build info: "idc_b200 <version> sm_100a ..." */
const char* idc_version(void);

/* Replaces `model.SIGGRAPHGenerator(dist=dist)` + `.cuda()` + `.eval()`
 * (data/colorize_image.py:221,230-232).  max_n = largest batch a forward may carry. */
int idc_create(int device, int max_n, int h, int w, unsigned flags, idc_ctx** out);

/* Plan-time options (replace the IDC_* environment switches of round 1; a library embedded in another process
 * must not read process-global state).  Call between idc_create and idc_finalize_weights / idc_adopt_weights;
 * a later call re-plans the launches.  -1 = automatic where it applies.
 *   "halo"          0 / 1 / 3   halo-tile A operand (one TMA tile per 64 input channels serves all 9 taps)
 *   "pairs"         0 / 1 / 2   cta_group::2 CTA pairs: never / large launches / always
 *   "mt"            1 / 2       128-pixel M-tiles per CTA tile on the <= 128-column layers
 *   "chunk_kb"      >= 1        k-blocks summed in TMEM before the FP32 round-to-nearest add (accuracy vs speed)
 *   "split_k"       >= 1        K slices per tile on launches that cannot fill the machine
 *   "split_pairs"   0 / 1       run the split-K (small batch) launches as CTA pairs
 *   "split_bn128"   0 / 1       128-column tiles on the split-K path (default 1: half the reduction traffic per CTA)
 *   "conv1_1_umma"  0 / 1       model1.0 on the tensor cores (default 1); 0 = the exact-FP32 CUDA-core kernel
 *   "host_pipe"     0 / 1      idc_forward_host: chunked copy/compute overlap for batches >= 8
 *   "pdl"           0 / 1       programmatic dependent launch between the kernels of one forward
 *   "side_dist"     0 / 1       batches <= 4: run the dist head (class + softmax) on a side stream / graph branch
 *   "tanh_scale"    110 / 100   regression head scale: tanh * 110 (model.py:175) or the Caffe nets' 100
 *                               (models/reference_model/deploy_nodist.prototxt:812-822, SURVEY q4)
 * Unknown names return IDC_ERR_KEY. */
int idc_set_option(idc_ctx* ctx, const char* name, int value);

/* Replaces one entry of `self.net.load_state_dict(state_dict)` (data/colorize_image.py:229).
 * key = reference state_dict key ("model1.0.weight", "model1.4.running_var", ...; conv OIHW,
 * deconv IOHW, model.py:13-108).  Extra keys accepted with IDC_FLAG_GLOBAL_HINTS:
 * "glob.{0,1,2,3}.weight/bias" + "glob.{0..3}.bn.*".  data is HOST memory. */
int idc_load_tensor(idc_ctx* ctx, const char* key, const void* data, int dtype, int ndim,
                    const int64_t* dims);

/* Packs every loaded tensor into the device-resident weight arena (K-major FP16 hi/lo
 * tiles for tcgen05, FP32 [K][Cout] for the SIMT engine; BatchNorm folded to scale/shift).
 * Fails with IDC_ERR_KEY if a required key is missing. */
int idc_finalize_weights(idc_ctx* ctx);

/* Device pointer + size of the packed arena: rank 0 broadcasts it once over NCCL
 * (SURVEY 8e); ranks != 0 call idc_adopt_weights() after receiving into it. */
int idc_weights_arena(idc_ctx* ctx, void** dev_ptr, size_t* bytes);
int idc_reserve_weights(idc_ctx* ctx);    /* allocate the arena without packing (receiver side) */
int idc_adopt_weights(idc_ctx* ctx);      /* mark a received arena as final                     */

/* Replaces `self.net.forward(img_l_mc, input_ab_mc, input_mask_mult, mask_cent)`
 * (data/colorize_image.py:263 / :308), batched.
 *   L_mc  [n,1,h,w]  L-50 in [-50,50]        ab [n,2,h,w] in [-110,110]
 *   mask  [n,1,h,w]  in [0,1]                maskcent: model.py:142
 *   glob  [n,316] or NULL: [313 ab histogram, 1 indicator, 1 mean saturation, 1 indicator]
 *         (data/colorize_image.py:452-463; deploy_nodist.prototxt:8-18)
 *   out_ab   [n,2,h,w]  tanh*110 (model.py:175).  NOTE the reference's dist=True return is
 *            tanh*110*110 (model.py:166-168, quirk q1); the Python mirror applies that.
 *   out_dist [n,529,h/4,w/4] or NULL: softmax(0.2*model_class(conv8_3)) BEFORE the nearest
 *            x4 upsample (model.py:160); requires IDC_FLAG_DIST.
 *   out_rgb  [n,h,w,3] uint8 or NULL: lab2rgb_transpose(L, out_ab)
 *            (data/colorize_image.py:20-28,264).
 * All pointers are DEVICE memory; asynchronous on `stream` (a cudaStream_t). */
int idc_forward(idc_ctx* ctx, int n, int h, int w, const float* L_mc, const float* ab,
                const float* mask, float maskcent, const float* glob, float* out_ab,
                float* out_dist, uint8_t* out_rgb, void* stream);

/* Same with HOST pointers (synchronous).  This is the call the reference-facing wrapper and bench.py's e2e leg use.
 * Batches <= 4 (the interactive click) replay ONE CUDA graph: a single H2D of the staged inputs, the kernels chained by
 * programmatic dependent launch, a single D2H of the results; batches >= 8 copy straight from / to pinned caller
 * buffers (pageable ones are staged) and overlap the copies with the first / last layer in image chunks.
 * L_mc may be NULL when idc_set_image has made the n L planes resident (then only the hints travel).
 * Results are bit-identical to idc_forward. */
int idc_forward_host(idc_ctx* ctx, int n, int h, int w, const float* L_mc, const float* ab,
                     const float* mask, float maskcent, const float* glob, float* out_ab,
                     float* out_dist, uint8_t* out_rgb);
/* Same + the reference's QUANTISED `self.output_ab` (row a11): out_abq [n,2,h,w] float64 =
 * rgb2lab(out_rgb)[1:] (`_set_out_ab_`, data/colorize_image.py:196-198,267; what the GUI and get_img_fullres read,
 * ui/gui_draw.py:280, :123-131), computed on the device from the just-quantised uint8 pixel, so the wrapper's
 * net_forward is ONE call and one round trip.  out_abq needs out_rgb; NULL = idc_forward_host. */
int idc_forward_host_q(idc_ctx* ctx, int n, int h, int w, const float* L_mc, const float* ab,
                       const float* mask, float maskcent, const float* glob, float* out_ab,
                       float* out_dist, uint8_t* out_rgb, double* out_abq);

/* The reference splits a session into `set_image` / `load_image` (the L plane, once per photo:
 * data/colorize_image.py:68-77, :186-189) and `net_forward(input_ab, input_mask)` (per click, :249).  idc_set_image is
 * the first half: it uploads the n mean-centred L planes [n,1,h,w] once; idc_forward_host(_q) calls with
 * L_mc == NULL and the same n then reuse them, so a click moves only the hints (3/4 of the input bytes).
 * n = 0 or L_mc = NULL forgets the image. */
int idc_set_image(idc_ctx* ctx, int n, int h, int w, const float* L_mc);

/* Page-locked host memory for the zero-copy click path: when every buffer handed to idc_forward_host(_q) with
 * n <= 4 comes from idc_host_alloc (or is otherwise pinned), the copy nodes of the click graph read / write the caller's
 * memory directly (no staging copy by the CPU); buffers laid out back to back -- [L | ab | mask (| glob)] and
 * [out_ab | out_rgb | out_abq] -- travel as one copy each way.  The graph is re-captured when the pointers change, so
 * keep the buffers for the lifetime of the session (LhnContext.click_buffers does). */
void* idc_host_alloc(size_t bytes);
int idc_host_free(void* p);

/* Interactive path: keep the 529-bin distribution of the last idc_forward_host on the device instead
 * of copying all of it back (8.7 MB at 256^2) -- the reference only ever reads one pixel of it per click
 * (`self.dist_ab[:, h, w]`, data/colorize_image.py:329).  With resident mode on, idc_forward_host runs the
 * dist head even when out_dist is NULL; idc_fetch_dist then copies dist[img, :, y4, x4] (529 floats) to
 * host memory, or the whole [529, h/4, w/4] plane when y4 < 0. */
int idc_set_dist_resident(idc_ctx* ctx, int on);
int idc_fetch_dist(idc_ctx* ctx, int img, int y4, int x4, float* out_host);

/* The click itself (BASELINE config 5; ui/gui_draw.py:126-142 -> predict_color / suggest_color): tell the context
 * BEFORE the forward which pixel (img, y4, x4) of the (h/4 x w/4) distribution grid the user clicked and how many colour
 * suggestions K (0 = none) the GUI will ask for.  The next idc_forward_host(_q) with n <= 4 and resident mode on then
 * also gathers that pixel's 529-bin pmf and clusters it (idc_ab_reccs with the default 8 restarts / 100 iterations /
 * PyTorch gamut grid) on the dist head's side branch of the click graph -- off the critical path -- and brings the 8 KB
 * answer back with the same graph launch: idc_fetch_dist / idc_ab_reccs for the same pixel (and K) then return from
 * pinned host memory without touching the device.  The coordinates live in mapped host memory and are read when the
 * graph runs, so moving the click never re-captures the graph.  y4 < 0 switches the mode off (one re-capture). */
int idc_set_click(idc_ctx* ctx, int img, int y4, int x4, int K);

/* Colour suggestions at one pixel of the resident distribution (SURVEY row f2; replaces
 * ColorizeImageTorchDist.get_ab_reccs, data/colorize_image.py:322-354: 25 000 inverse-CDF samples of
 * dist_ab[:, h, w] -> sklearn KMeans(K) -> centres ordered by occupancy).  Computed as the sample-size ->
 * infinity limit of that procedure: deterministic weighted k-means over the 529 gamut points with the pmf
 * as weights (seeds: heaviest bin, then argmax w*d^2; FP64 Lloyd iterations until the assignment is stable
 * or max_iter); n_init restarts run side by side (restart v seeds from the bin of weight-rank v) and the one
 * with the lowest inertia wins (sklearn's n_init; 1 <= n_init <= 16).  pts_host: [529][2] ab coordinates of the bins, or NULL for the PyTorch wrapper's grid
 * (bin i = (g[i % 23], g[i / 23]), g = -110..110 step 10, :283).  Outputs (host): centers [K][2], conf [K]
 * (cluster mass, descending; may be NULL), iters_out (Lloyd iterations used; may be NULL).  1 <= K <= 32. */
int idc_ab_reccs(idc_ctx* ctx, int img, int y4, int x4, int K, int max_iter, int n_init, const float* pts_host,
                 float* centers_host, float* conf_host, int* iters_out);
/* Same clustering for a caller-supplied pmf (host, 529 floats, need not be normalised); no ctx needed. */
int idc_ab_reccs_pmf(int device, const float* pmf_host, int K, int max_iter, int n_init, const float* pts_host,
                     float* centers_host, float* conf_host, int* iters_out);

/* Caffe-spec 313-bin head (SURVEY row a14; models/reference_model/deploy_nopred.prototxt:651-850, weight
 * injection data/colorize_image.py:405-413).  With IDC_FLAG_CAFFE313 every forward also runs the
 * hyper-column (conv3_pred + conv4..7_pred + conv8_pred, ReLU) and pred_313 (1x1 -> 313 logits at h/4).
 * Extra state_dict keys: "caffe.conv{3..8}_pred.{weight,bias}" (conv3/8: [384,256,3,3]; conv4..7: Caffe
 * Deconvolution [512,384,4,4]), "caffe.pred_313.{weight,bias}" [313,384,1,1], "caffe.pts_in_hull" [313,2].
 *   idc_caffe313_pred_ab:    two grouped bilinear x2 deconvs (kernel [[.25,.5,.25,0],[.5,1,.5,0],[.25,.5,.25,0],0])
 *                            -> softmax(T * logits) -> annealed mean over the 313 bin centres = pred_ab [n,2,h,w]
 *                            (DEVICE pointer; T = 2.6 in the reference, :827-848).
 *   idc_caffe313_dist_pixel: dist_ab_S[:, y, x] = softmax(S * upsampled logits) at ONE full-resolution
 *                            pixel (S = 0.2, :808-820) -> 313 floats in HOST memory. */
int idc_caffe313_pred_ab(idc_ctx* ctx, int n, float T, float* out_ab, void* stream);
int idc_caffe313_dist_pixel(idc_ctx* ctx, int img, int y, int x, float S, float* out313_host);

/* Stand-alone post-process: lab2rgb_transpose (data/colorize_image.py:20-28).
 * L [n,1,h,w] in [0,100] (NOT mean-centred), ab [n,2,h,w] -> rgb [n,h,w,3] uint8. DEVICE ptrs. */
int idc_lab2rgb_u8(int device, int n, int h, int w, const float* L, const float* ab,
                   uint8_t* rgb, void* stream);

/* f1 (steps either side of the network), float64 like the reference's numpy/skimage/scipy path; DEVICE ptrs.
 * idc_rgb2lab_f64:      skimage color.rgb2lab of uint8 RGB [n,h,w,3] -> Lab planes [n,3,h,w] float64
 *                       (data/colorize_image.py:31-36, :172-178 image prep, :196-198 _set_out_ab_).
 * idc_zoom_lab2rgb_u8:  get_img_fullres (:123-131): scipy.ndimage.zoom(order=1) of ab [2,h_in,w_in] to
 *                       [h,w], then lab2rgb_transpose with the full-resolution L [h,w] -> uint8 [h,w,3]. */
int idc_rgb2lab_f64(int device, int n, int h, int w, const uint8_t* rgb, double* lab, void* stream);
/* f3: global statistics of a reference image (models/global_model/global_stats.prototxt:1-244; NNEncLayer with
 * NN=1, caffe_files/caffe_traininglayers.py:161-196; usage DemoGlobalHistogramTransfer.ipynb:176-182):
 * uint8 RGB [h,w,3] (h,w multiples of 4) + the 313 ab bin centres [313,2] -> out[316] =
 * [313-bin histogram of the 4x4-pooled ab, 1, mean HSV saturation, 1] = the `glob` input of idc_forward. DEVICE ptrs. */
int idc_global_stats(int device, int h, int w, const uint8_t* rgb, const float* pts313, float* out316, void* stream);
int idc_zoom_lab2rgb_u8(int device, int h_in, int w_in, const double* ab, int h, int w, const double* L_full,
                        uint8_t* rgb, void* stream);

/* f1, image-load side (data/colorize_image.py:52-66): cv2.resize(im, (w_dst, h_dst)) of a uint8 [h,w,3] image with
 * OpenCV's default INTER_LINEAR -- the 8-bit path of OpenCV is fixed-point arithmetic and is restated integer for
 * integer (bit-identical to cv2, incl. the exact-2x shortcut to area averaging).  DEVICE ptrs. */
int idc_resize_u8_linear(int device, int h_src, int w_src, const uint8_t* src, int h_dst, int w_dst, uint8_t* dst,
                         void* stream);
/* f1, GUI display step (ui/gui_draw.py:280-283): cv2.resize(ab [2,h_in,w_in] float64, (w,h), INTER_CUBIC), concatenated
 * with the window-size L [h,w] float64, skimage lab2rgb, clip, x255, truncating cast -> uint8 [h,w,3].  DEVICE ptrs. */
int idc_cubic_lab2rgb_u8(int device, int h_in, int w_in, const double* ab, int h, int w, const double* L, uint8_t* rgb,
                         void* stream);

/* ---- introspection / test hooks (used by tests/, never by the product path) ---- */
/* Copy a named activation ("conv1_2", "a8_1", ... see DESIGN.md) of the LAST forward to
 * out [n,C,H,W] FP32 device memory; *c,*h,*w receive its shape. */
int idc_get_activation(idc_ctx* ctx, const char* name, float* out_nchw, size_t out_floats,
                       int* c, int* h, int* w);
/* Overwrite a named activation from [n,C,H,W] FP32 device memory, then run ONE op by name. */
int idc_set_activation(idc_ctx* ctx, const char* name, int n, const float* in_nchw);
int idc_run_op(idc_ctx* ctx, const char* op_name, int n, void* stream);
int idc_num_ops(idc_ctx* ctx);
const char* idc_op_name(idc_ctx* ctx, int i);
/* Per-op device timing (CUDA events on the forward's stream, recorded between the op launches).
 * idc_set_profiling(ctx, 1) starts accumulating over subsequent forwards; idc_get_profile
 * synchronises, writes the MEAN milliseconds per forward of slot i into ms[i] (slot 0 = fused
 * pack+conv1_1, slots 1..num_ops = the ops in idc_op_name order, last slot = heads/post) and resets.
 * Returns the number of slots (num_ops + 2) or <0. */
int idc_set_profiling(idc_ctx* ctx, int enable);
int idc_get_profile(idc_ctx* ctx, float* ms, int max_slots);
/* FLOPs (2*MACs) of op i for ONE image (0 for out-of-range i) */
double idc_op_flops(idc_ctx* ctx, int i);
/* kernels launched by the last forward (gpu_launches in bench.py) */
int idc_last_launch_count(idc_ctx* ctx);
/* FLOPs (2*MACs, conv+deconv) of one image at the ctx geometry; includes model_class iff DIST */
double idc_flops_per_image(idc_ctx* ctx);

const char* idc_last_error(idc_ctx* ctx);
int idc_destroy(idc_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* IDC_B200_H_ */
