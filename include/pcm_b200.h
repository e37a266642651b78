/*
 * pcm_b200.h -- C ABI of the B200-native PixelClassification (PC) masker hot path.
 *
 * Drop-in boundary for the per-frame path of the reference
 * materight/non-rigid-object-tracking:
 *     maskers/pixel_classification.py:45-126   PixelClassificationNonRigidMasker.update
 *     maskers/pixel_classification.py:230-277  compileSaliencyMap / getFeatures (numba)
 *     maskers/pixel_classification.py:294-309  buildFramesParameter (cv.cvtColor)
 *     benchmark.py:8-14                        computeBenchmark (IoU)
 * The reference binds its only native component the same way
 * (prim/__init__.py:7-38 -> ctypes -> extern "C" rp(), prim/src/rp_py.cpp:7-23);
 * INTEGRATION.md shows the ctypes stub a maintainer adds for this library.
 *
 * Conventions
 *   - plain pointers and sizes only; no ownership transfer; every function
 *     returns 0 on success or a negative PCM_E_* code, and the message is
 *     available from pcm_last_error() (thread-local).
 *   - "host" entry points take HOST buffers and include the host<->device
 *     copies; "_device" entry points take DEVICE buffers, enqueue on the
 *     handle's stream and do not synchronise.
 *   - images are 8-bit, BGR interleaved (OpenCV layout), rows `stride` bytes apart.
 *   - there is NO CPU fallback: without a CUDA device pcm_create fails.
 */
#ifndef PCM_B200_H
#define PCM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCM_ABI_VERSION 1

enum {
    PCM_OK = 0,
    PCM_E_INVALID = -1,      /* bad argument */
    PCM_E_CUDA = -2,         /* CUDA runtime error */
    PCM_E_STATE = -3,        /* call order (e.g. model before features) */
    PCM_E_LIMIT = -4,        /* exceeds a documented limit */
    PCM_E_LABEL = -5         /* label outside [0, n_labels) */
};

/* colour-space ids of the `features` token (pixel_classification.py:301-308) */
enum { PCM_SPACE_RGB = 0 /* raw BGR planes */, PCM_SPACE_HSV = 1, PCM_SPACE_LAB = 2 };

typedef struct pcm_handle pcm_handle;

/* ---- lifetime -------------------------------------------------------- */

int pcm_abi_version(void);
const char* pcm_last_error(void);

/* One handle per masker instance (= per tracked target, main.py:138-144). */
int pcm_create(int device, pcm_handle** out);
void pcm_destroy(pcm_handle* h);

/* Enqueue on an existing CUDA stream (cudaStream_t passed as void*; NULL is the
 * legacy default stream) instead of the handle's own non-blocking stream;
 * pcm_use_own_stream switches back. */
int pcm_set_stream(pcm_handle* h, void* cuda_stream);
int pcm_use_own_stream(pcm_handle* h);
/* The stream work is currently enqueued on (cudaStream_t as void*), e.g. to record timing events on the
 * handle's private stream from another runtime. */
int pcm_get_stream(const pcm_handle* h, void** cuda_stream_out);
/* Waits for the stream; reports (once) an out-of-range label met by ANY update queued since the last check. */
int pcm_synchronize(pcm_handle* h);

/* ---- configuration (config.yaml `params.features`, :300-308) ---------- */

/* "8 hsv_lab" -> n_neighbors = 8, space_ids = {HSV, LAB}.  Must precede
 * pcm_add_model.  Limits: 1 <= n_neighbors <= 16, 1 <= n_spaces <= 3. */
int pcm_set_features(pcm_handle* h, int n_neighbors, int n_spaces, const int* space_ids);

/* Number of features per pixel F = 3 * (1 + 8 n) * n_spaces (:252-261). */
int pcm_num_features(const pcm_handle* h);

/* ---- models (addModel :166-228; training itself stays with the caller) -- */

/* Append one fitted random forest (sklearn RandomForestClassifier arrays,
 * estimators_ order, nodes of tree t at [tree_offsets[t], tree_offsets[t+1])):
 *   feature[i]    column of X tested at node i            (tree_.feature)
 *   threshold[i]  float64 split value on X/255            (tree_.threshold)
 *   left/right[i] child node ids within the tree, -1 leaf (tree_.children_*)
 *   value1[i]     class-1 fraction at node i              (tree_.value[i,0,1])
 * Thresholds are collapsed to integers here (x_f32 <= thr  <=>  v <= t), so
 * scoring is bit-exact against predict_proba (:80,:82).
 * Returns the model index in *model_index. */
int pcm_add_model(pcm_handle* h, int n_frame, int n_trees, const int64_t* tree_offsets,
                  const int32_t* feature, const double* threshold,
                  const int32_t* left, const int32_t* right, const double* value1,
                  int* model_index);

/* Attach the novelty detector of a model: PCA mean_[F], components_[0][F]
 * (n_components == 1, config.yaml:27) (:205-213).  Same as pcm_set_novelty_k with n_components = 1. */
int pcm_set_novelty(pcm_handle* h, int model_index, const double* mean, const double* component, int n_features);

/* The novelty detector of a PCA with several components (params.n_components, :203-213): mean_[F] and
 * components_[n_components][F], row-major, as scikit-learn stores them.  1 <= n_components <= PCM_MAX_PCA_COMPONENTS
 * (PCM_E_INVALID below, PCM_E_LIMIT above).  A frame whose current or next model has two or more components computes
 * the reconstruction error in a kernel of its own (profile id 7); rank-1 models keep the score kernel's in-line pass. */
#define PCM_MAX_PCA_COMPONENTS 8
int pcm_set_novelty_k(pcm_handle* h, int model_index, const double* mean, const double* components, int n_components,
                      int n_features);

int pcm_num_models(const pcm_handle* h);

/* ---- per-frame hot path ------------------------------------------------ */

/* The reference's bbox enlargement + numpy slice clamping (:49-51):
 * rect_out = {x, y, w, h} of the crop actually processed. */
int pcm_crop_rect(const int bbox_xywh[4], int frame_h, int frame_w, int rect_out[4]);

typedef struct pcm_update_params {
    int32_t model_cur;           /* current model index */
    int32_t model_next;          /* next model to blend with, or -1 (:81) */
    double w_cur;                /* np.average weights (:87): 1 - tmp/span */
    double w_next;               /*                            tmp/span    */
    int32_t novelty;             /* params.novelty_detection (:57) */
    int32_t dilation_kernel;     /* params.dilation_kernel (:112) */
    double outlier_threshold;    /* novelty_det[cur].threshold (:108) */
    double prior_weight;         /* params.prior_weight (:107) */
} pcm_update_params;

/* One `update()` (:45-112) on HOST buffers, synchronous:
 *   frame     H x W x 3 BGR, rows frame_stride bytes apart; not modified
 *   rect      crop {x, y, w, h} from pcm_crop_rect
 *   labels    h*w int32 over-segmentation labels of the crop, values in [0, n_labels);
 *             n_labels <= 0: taken as max(label) + 1 (found while the map is staged;
 *             only without priors).  Label chunks identical to the previous call's are
 *             not re-sent to the device.
 *   priors    n_labels float32 (computePriors :129-163) or NULL for all -1
 *   mask      first byte of the channel to write (the reference writes channel 2
 *             of an H x W x 3 image: mask + 2, mask_pixel_stride = 3); only the
 *             crop rectangle is written (overwrite, then dilation, :246,:112)
 * Host->device copies of frame crop / labels / priors and the device->host copy
 * of the mask are inside this call. */
int pcm_update(pcm_handle* h, const uint8_t* frame, int frame_h, int frame_w, int64_t frame_stride,
               const int rect[4], const int32_t* labels, int n_labels, const float* priors,
               const pcm_update_params* params,
               uint8_t* mask, int64_t mask_row_stride, int64_t mask_pixel_stride);

/* labels == NULL: continue from the preceding pcm_quickshift, pcm_slic_gpu or pcm_felzenszwalb_gpu on this handle -- the label map
 * AND the crop pixels are the ones that call left on the device (`frame` and `rect` must be
 * the same as in that call; the frame is not read again).  n_labels is ignored. */

/* pcm_update keeps the previous call's label map (pinned host copy + device copy) and re-sends
 * only the 1 MiB chunks whose bytes changed.  on = 0 switches that off: every call uploads the
 * whole map (default: on). */
int pcm_set_label_cache(pcm_handle* h, int on);

/* labels == NULL with no pcm_quickshift / pcm_slic_gpu / pcm_felzenszwalb_gpu pending: the label map the previous pcm_update left on the device is used
 * again (same crop size required; n_labels is ignored).  The caller vouches that the map has not changed -- the
 * plugin does this when its over-segmentation provider hands back the very same read-only array. */

/* Page-lock a long-lived caller buffer (cudaHostRegister, portable) so that pcm_update / pcm_iou copy a frame or truth
 * image that lies inside it straight from the caller's memory instead of staging it through the handle's pinned
 * buffers.  The range must stay allocated until pcm_host_unregister(p) (same start address). */
int pcm_host_register(void* p, size_t bytes);
int pcm_host_unregister(void* p);

/* Same work on DEVICE buffers, asynchronous on the handle's stream.
 * d_mask is a dense plane (pixel stride 1) of frame_h x frame_w, rows
 * mask_row_stride bytes apart; only the crop rectangle is written. */
int pcm_update_device(pcm_handle* h, const uint8_t* d_frame, int frame_h, int frame_w, int64_t frame_stride,
                      const int rect[4], const int32_t* d_labels, int n_labels, const float* d_priors,
                      const pcm_update_params* params,
                      uint8_t* d_mask, int64_t mask_row_stride);

/* computeBenchmark (benchmark.py:8-14): counts[0] = #(mask!=0 && truth!=0),
 * counts[1] = #(mask!=0 || truth!=0) over h x w; the caller forms the float64
 * quotient (NaN on an empty union, like numpy).  truth_channels = 1 (gray) or
 * 3 (BGR frame: converted with cv.cvtColor(BGR2GRAY) arithmetic, main.py:285). */
int pcm_iou(pcm_handle* h, const uint8_t* mask, int64_t mask_row_stride, int64_t mask_pixel_stride,
            const uint8_t* truth, int64_t truth_row_stride, int truth_channels,
            int height, int width, int64_t counts[2]);

/* Device variant: dense mask plane and truth on the device; counts are added
 * into d_counts[2] (int64, caller zeroes), asynchronous. */
int pcm_iou_device(pcm_handle* h, const uint8_t* d_mask, int64_t mask_row_stride,
                   const uint8_t* d_truth, int64_t truth_row_stride, int truth_channels,
                   int height, int width, int64_t* d_counts);

/* ---- over-segmentation of the crop (:70-71), SURVEY.md §8 row f-1 ----------- */

/* skimage.segmentation.quickshift(crop, kernel_size, max_dist, ratio, random_seed) of
 * scikit-image 0.17.2 (environment.yaml:12) on the crop `rect` of a HOST frame:
 * sRGB->Lab (float64; the BGR channel order is taken as it comes, like the reference does),
 * window densities, nearest-higher-density parent, links longer than max_dist cut, labels
 * numbered like np.unique(root, return_inverse=True).
 *   noise       h*w float64 = RandomState(random_seed).normal(scale=1e-5, size=(h, w)), the
 *               tie-breaking noise of _quickshift_cy.pyx, or NULL to reuse the noise of the
 *               previous call with the same crop size
 *   labels_out  h*w int32 on the host, or NULL when only the device-resident map is needed
 *               (pcm_update with labels == NULL)
 *   n_labels_out  number of segments
 * Limits: ceil(3 * kernel_size) <= 15.  Synchronous. */
int pcm_quickshift(pcm_handle* h, const uint8_t* frame, int frame_h, int frame_w, int64_t frame_stride,
                   const int rect[4], double ratio, double kernel_size, double max_dist,
                   const double* noise, int32_t* labels_out, int* n_labels_out);

/* Device variant: d_frame / d_noise (may be NULL: no noise) / d_labels_out (h*w int32, may be
 * NULL) are device pointers; waits for the stream to return the segment count.
 * Limits: those of pcm_quickshift, and frame_stride >= 3 * frame_w. */
int pcm_quickshift_device(pcm_handle* h, const uint8_t* d_frame, int frame_h, int frame_w, int64_t frame_stride,
                          const int rect[4], double ratio, double kernel_size, double max_dist,
                          const double* d_noise, int32_t* d_labels_out, int* n_labels_out);

/* The label maps of n crops of a device-resident clip in one call (the sweep computes the maps of a whole clip before
 * its sequences start, pixel_classification.py:71 once per frame): crop k = rects[4k .. 4k+3] of the frame at
 * d_frames + frame_index[k] * frame_bytes, its map written at d_labels_out + label_offsets[k] (int32 elements), its
 * segment count at n_labels_out[k] (host).  Exactly n calls of pcm_quickshift_device -- one wait per crop included, so
 * that the stream never holds more than one crop's launches -- without returning to the caller in between. */
int pcm_quickshift_device_batch(pcm_handle* h, int n, const uint8_t* d_frames, int64_t frame_bytes, const int32_t* frame_index,
                                int frame_h, int frame_w, int64_t frame_stride, const int32_t* rects, double ratio,
                                double kernel_size, double max_dist, const double* d_noise, int32_t* d_labels_out,
                                const int64_t* label_offsets, int32_t* n_labels_out);

/* skimage.segmentation.felzenszwalb(crop, scale, sigma, min_size) of scikit-image 0.17.2 (:72-73) on
 * the crop `rect` of a HOST frame.  HOST code (no handle, no device): the reference the GPU variant
 * pcm_felzenszwalb_gpu is tested against.  Edges of equal cost are processed in a fixed order
 * (right, down, down-right, up-right; raster order within each).
 *   kernel      2 * kernel_radius + 1 Gaussian weights (scipy's _gaussian_kernel1d), or NULL to
 *               compute them from sigma
 *   labels_out  h*w int32, labels numbered like np.unique(root, return_inverse=True) */
int pcm_felzenszwalb(const uint8_t* frame, int frame_h, int frame_w, int64_t frame_stride, const int rect[4],
                     double scale, double sigma, int min_size, const double* kernel, int kernel_radius,
                     int32_t* labels_out, int* n_labels_out);

/* skimage.segmentation.slic(crop, n_segments, compactness, sigma, max_iter = 10, start_label) of scikit-image 0.17.2
 * (:74-75: n_segments = 250, compactness = 10, sigma = 1, start_label = 0) on the crop `rect` of a HOST frame: Gaussian,
 * rgb2lab, k-means from a regular seed grid, connectivity enforcement.  HOST code (no handle, no device), like
 * pcm_felzenszwalb; parity pinned only against oracle/slic_oracle.py (scikit-image is not available here).
 *   kernel      2 * kernel_radius + 1 Gaussian weights (scipy's _gaussian_kernel1d), or NULL to compute them from sigma
 *   labels_out  h*w int32, labels start_label .. ; n_labels_out = largest label + 1 */
int pcm_slic(const uint8_t* frame, int frame_h, int frame_w, int64_t frame_stride, const int rect[4], int n_segments,
             double compactness, double sigma, const double* kernel, int kernel_radius, int max_iter, int start_label,
             int32_t* labels_out, int* n_labels_out);

/* pcm_slic on the GPU: the same labels and count as pcm_slic for the same arguments (DESIGN.md §10).  Only rgb2lab may
 * differ from the host code, by at most 1e-12 on the image the k-means sees, because CUDA's pow / cbrt are not glibc's.
 * The crop of a HOST frame is staged like pcm_quickshift's, and the label map stays on the device: pcm_update with
 * labels == NULL (same frame and rect) continues from it.  Synchronous.
 *   kernel      2 * kernel_radius + 1 Gaussian weights on the host, or NULL to compute them from sigma as pcm_slic does
 *   labels_out  h*w int32 on the host, or NULL when only the device-resident map is needed
 * Limits: crop of at most 2^28 pixels; n_segments >= 1, compactness > 0, max_iter >= 0, start_label >= 0. */
int pcm_slic_gpu(pcm_handle* h, const uint8_t* frame, int frame_h, int frame_w, int64_t frame_stride, const int rect[4],
                 int n_segments, double compactness, double sigma, const double* kernel, int kernel_radius, int max_iter,
                 int start_label, int32_t* labels_out, int* n_labels_out);

/* Device variant: d_frame and d_labels_out (h*w int32, may be NULL) are device pointers, `kernel` is on the host; waits
 * for the stream to return the segment count. */
int pcm_slic_device(pcm_handle* h, const uint8_t* d_frame, int frame_h, int frame_w, int64_t frame_stride, const int rect[4],
                    int n_segments, double compactness, double sigma, const double* kernel, int kernel_radius, int max_iter,
                    int start_label, int32_t* d_labels_out, int* n_labels_out);

/* The SLIC maps of n crops of a device-resident clip in one call, laid out like pcm_quickshift_device_batch's: exactly n
 * calls of pcm_slic_device without returning to the caller in between. */
int pcm_slic_device_batch(pcm_handle* h, int n, const uint8_t* d_frames, int64_t frame_bytes, const int32_t* frame_index,
                          int frame_h, int frame_w, int64_t frame_stride, const int32_t* rects, int n_segments, double compactness,
                          double sigma, const double* kernel, int kernel_radius, int max_iter, int start_label,
                          int32_t* d_labels_out, const int64_t* label_offsets, int32_t* n_labels_out);

/* Parity tap: the device connectivity enforcement of pcm_slic_gpu on a caller's centre map `nearest` (width x height int32,
 * host), with the caller's min_size / max_size (pcm_slic uses (long long)(0.5 s) and (long long)(3 s) for the segment size
 * s = h*w / n_segments).  labels_out: width*height int32 (host); n_labels_out = largest label + 1. */
int pcm_slic_connectivity(pcm_handle* h, const int32_t* nearest, int width, int height, long long min_size, long long max_size,
                          int start_label, int32_t* labels_out, int* n_labels_out);

/* Parity tap: the stage results of the last pcm_slic_gpu / pcm_slic_device on the handle, each h*w pixels of that crop:
 * smoothed (3 float64 per pixel: /255 and the Gaussian), image (3 float64: rgb2lab / compactness, what the k-means sees),
 * nearest (int32: the centre map after the last k-means iteration).  NULL skips a stage.  PCM_E_STATE before any SLIC. */
int pcm_slic_debug_last(pcm_handle* h, double* smoothed, double* image, int32_t* nearest);

/* Parity tap: the cost-ordered merge, union-find and min-size passes of pcm_felzenszwalb on a caller-provided
 * edge list (n_edges edges a[i]-b[i] with non-negative cost[i]; `scale` is the k of k/|C|, already on the scale
 * of the costs).  Same host code as pcm_felzenszwalb after its edge construction; checked against the
 * Felzenszwalb-Huttenlocher code the reference vendors (prim/src/FelzenSegment/segment-graph.h:48-81,
 * segment_image_index.h:85-91) in tests/test_felzenszwalb_ref.py.  labels_out: n_vertices int32. */
int pcm_felzenszwalb_graph(int n_vertices, int n_edges, const int32_t* a, const int32_t* b, const double* cost,
                           double scale, int min_size, int32_t* labels_out, int* n_labels_out);

/* pcm_felzenszwalb on the GPU: the same labels and count as pcm_felzenszwalb for the same arguments (DESIGN.md §9).  The
 * cost-ordered merge runs in rounds that decide, in parallel, only edges whose outcome is already certain, so the partition
 * is the host's exactly.  The crop of a HOST frame is staged like pcm_quickshift's, and the label map stays on the device:
 * pcm_update with labels == NULL (same frame and rect) continues from it.  Synchronous.
 *   kernel      2 * kernel_radius + 1 Gaussian weights on the host, or NULL to compute them from sigma as pcm_felzenszwalb does
 *   labels_out  h*w int32 on the host, or NULL when only the device-resident map is needed
 * Limits: crop of at most 2^28 pixels; kernel_radius >= 0 with a kernel; frame_stride >= 3 * frame_w. */
int pcm_felzenszwalb_gpu(pcm_handle* h, const uint8_t* frame, int frame_h, int frame_w, int64_t frame_stride, const int rect[4],
                         double scale, double sigma, int min_size, const double* kernel, int kernel_radius,
                         int32_t* labels_out, int* n_labels_out);

/* Device variant: d_frame and d_labels_out (h*w int32, may be NULL) are device pointers, `kernel` is on the host; waits
 * for the stream to return the segment count. */
int pcm_felzenszwalb_device(pcm_handle* h, const uint8_t* d_frame, int frame_h, int frame_w, int64_t frame_stride,
                            const int rect[4], double scale, double sigma, int min_size, const double* kernel, int kernel_radius,
                            int32_t* d_labels_out, int* n_labels_out);

/* The Felzenszwalb maps of n crops of a device-resident clip in one call, laid out like pcm_quickshift_device_batch's:
 * the same maps and counts as n calls of pcm_felzenszwalb_device.  The crops run in one batched pass: consecutive crops
 * are grouped into chunks of at most 2^23 pixels (a larger crop is a chunk of its own), and each chunk is one graph of
 * disjoint pieces whose merge rounds serve all its crops at once, so it takes as many rounds as its slowest crop.  Every
 * crop is checked before any work is queued; the counts come back with one wait for the whole batch.  Like every
 * over-segmentation call (n > 0), it ends a pending pcm_update(labels == NULL) handoff. */
int pcm_felzenszwalb_device_batch(pcm_handle* h, int n, const uint8_t* d_frames, int64_t frame_bytes, const int32_t* frame_index,
                                  int frame_h, int frame_w, int64_t frame_stride, const int32_t* rects, double scale, double sigma,
                                  int min_size, const double* kernel, int kernel_radius, int32_t* d_labels_out,
                                  const int64_t* label_offsets, int32_t* n_labels_out);

/* Parity tap: the device twin of pcm_felzenszwalb_graph (same arguments, same validation; a, b, cost and labels_out on the
 * host): the sort, the two passes in rounds and the labelling of pcm_felzenszwalb_gpu on a caller's edge list. */
int pcm_felzenszwalb_graph_gpu(pcm_handle* h, int n_vertices, int n_edges, const int32_t* a, const int32_t* b,
                               const double* cost, double scale, int min_size, int32_t* labels_out, int* n_labels_out);

/* Parity tap: for the last pcm_felzenszwalb_gpu / _device / _device_batch / _graph_gpu call on the handle, smoothed (h*w*3
 * float64 of that call's last crop: /255 and the Gaussian; NULL skips it, and it must be NULL after the graph tap) and
 * rounds[2] (int32: the rounds of the merge pass and of the min-size pass -- after a batch, the largest over its crops;
 * NULL skips it).  PCM_E_STATE before any such call. */
int pcm_felzenszwalb_debug_last(pcm_handle* h, double* smoothed, int32_t* rounds);

/* ---- a whole sequence of frames in one call (main.py:280-343 for one target) ---- */

/* One frame of a device-resident sequence: [priors from SIFT matches] -> [clear the mask plane] -> update -> [IoU].
 * Every pointer is a device pointer; 0 / NULL switches the optional step off. */
typedef struct pcm_frame_job {
    const uint8_t* d_frame;        /* frame_h x frame_w x 3 BGR */
    int32_t rect[4];               /* crop {x, y, w, h} from pcm_crop_rect */
    const int32_t* d_labels;       /* over-segmentation of the crop */
    int32_t n_labels;
    int32_t clear_mask;            /* a fresh mask per frame (main.py:286): 1 = zero the whole plane before the update;
                                    * 2 = leave the plane alone and let the IoU step read it as zero outside `rect`
                                    * (same counts, no memset; the plane is then scratch outside the current crop) */
    pcm_update_params params;
    /* pcm_prior_device before the update (skipped when d_priors_out is NULL): the previous frame's mask is read from
     * the mask plane at prev_rect, BEFORE the plane is cleared */
    const float* d_pts_prev; const uint8_t* d_des_prev; int32_t n_prev; int32_t prev_rect[4];
    const float* d_pts; const uint8_t* d_des; int32_t n_cur; int32_t reserved;
    float* d_priors_out;           /* n_labels float32: filled by the prior step and used by the update */
    const float* d_priors;         /* priors for the update when there is no prior step (NULL: all -1) */
    /* pcm_iou_device after the update (skipped when d_truth is NULL) */
    const uint8_t* d_truth; int64_t truth_stride; int32_t truth_channels; int32_t reserved2;
    int64_t* d_counts;             /* two int64, caller-zeroed */
} pcm_frame_job;

/* Enqueue n_jobs frames back to back on the handle's stream (no host synchronisation in between or at the end):
 * the per-frame work of pcm_prior_device / pcm_update_device / pcm_iou_device, issued from native code so that a
 * sequence costs one call.  d_mask: dense frame_h x frame_w plane shared by the frames. */
int pcm_run_frames(pcm_handle* h, int frame_h, int frame_w, int64_t frame_stride, uint8_t* d_mask, int64_t mask_row_stride,
                   const pcm_frame_job* jobs, int n_jobs);

/* ---- SIFT-match prior (computePriors :129-163), SURVEY.md §8 row f-2 -------- */

/* Priors of one frame from the SIFT keypoints / descriptors the caller detected with OpenCV (host, once per clip
 * frame) and uploaded: d_pts* = (x, y) float32 pairs in crop coordinates, d_des* = 128 uint8 per keypoint (OpenCV's
 * float32 descriptors hold integers 0..255), 16-byte aligned.
 *   previous crop: all keypoints of the UNMASKED detection; the mask filter of detectAndCompute(prev, prevMask) --
 *                  keep mask[(int)(y + 0.5f)][(int)(x + 0.5f)] != 0 -- is applied here.  d_prev_mask points at the
 *                  previous crop's top-left pixel inside the (device) mask plane, rows prev_mask_stride apart.
 *   matching:      EXACT 2-nearest neighbours in squared L2 (ties to the smaller index) where the reference asks
 *                  FLANN's randomised kd-trees for approximate ones; ratio test m.distance < 0.7 * n.distance on the
 *                  float32 square roots (:147); displacement filter dist <= np.percentile(dist, 90) (:155-157)
 *   output:        d_priors[n_labels] = -1, and +1 for labels[int(y)][int(x)] of every surviving current keypoint (:159-161)
 * Fewer than one previous or two current keypoints: all -1, like the reference (:139).  Asynchronous. */
int pcm_prior_device(pcm_handle* h, const float* d_pts_prev, const uint8_t* d_des_prev, int n_prev,
                     const uint8_t* d_prev_mask, int64_t prev_mask_stride, int prev_w, int prev_h,
                     const float* d_pts, const uint8_t* d_des, int n_cur, const int32_t* d_labels, int crop_w, int crop_h,
                     int n_labels, float* d_priors);

/* ---- training (addModel :166-228), SURVEY.md §8 row f-3 ------------------- */

/* Grow, on the GPU, the trees that scikit-learn 1.9's
 *     RandomForestClassifier(random_state, n_estimators, max_depth).fit(X / 255, y)      (:199-200)
 * grows -- node for node, threshold for threshold (tests compare the arrays with scikit-learn's tree_).
 *   X            n_rows x n_features int16, row-major, raw feature values v in [-1, 255] as
 *                pcm_gather_features returns them (the reference trains on X / 255, :196), or NULL to reuse the
 *                rows that the previous call with the same non-zero rows_id left on the device
 *   y            n_rows class labels 0 / 1 (both present)
 *   counts       n_trees x n_rows bootstrap counts (np.bincount of RandomState(tree seed).randint(0, n, n),
 *                sklearn/ensemble/_forest.py:148-153), each <= 127
 *   rand_states  n_trees splitter seeds (RandomState(tree seed).randint(0, 2**31 - 1), tree/_splitter.pyx:155)
 *   max_features features drawn per node: max(1, int(sqrt(n_features))) for the reference's default
 *   node_capacity  stride of the per-tree outputs; 2^(max_depth+1) - 1 always suffices
 * Outputs, tree t at [t * node_capacity, ...): node_count[t]; feature (-2 = leaf), threshold (-2.0 = leaf),
 * left / right (-1 = leaf), value1 = class-1 fraction of the node, n_node_samples (may be NULL), nodes in
 * scikit-learn's depth-first order.  The arrays feed pcm_add_model unchanged.  Synchronous.
 * Limits: n_rows < 2^24, n_features <= 1176, max_depth <= 24. */
int pcm_fit_forest(pcm_handle* h, const int16_t* X, const uint8_t* y, int n_rows, int n_features, long long rows_id,
                   int n_trees, int max_depth, int max_features, const uint8_t* counts, const uint32_t* rand_states,
                   int node_capacity, int32_t* node_count, int32_t* feature, double* threshold,
                   int32_t* left, int32_t* right, double* value1, int32_t* n_node_samples);

/* Upload a training-row set (as for pcm_fit_forest) without fitting; it stays resident under rows_id != 0. */
int pcm_fit_rows(pcm_handle* h, const int16_t* X, const uint8_t* y, int n_rows, int n_features, long long rows_id);

/* Novelty detector of addModel (:203-213: PCA(n_components=k).fit(X[labels == 1]), then the L1 reconstruction
 * error of every training row) on the RESIDENT rows `rows_id`:
 *   pcm_pca_moments      gram[F*F] = sum over class-1 rows of v v^T, sums[F] = sum of v (raw integer feature values,
 *                        exact), n_class1.  The caller forms sklearn's covariance (decomposition/_pca.py, solver
 *                        covariance_eigh) and takes its leading eigenvectors (pcm/train.py: numpy.linalg.eigh).
 *   pcm_pca_residuals    err[n_rows] = sum_f |x_f - (t c_f + mean_f)|, t = x.c - mean.c, x = v / 255 (:208-211) for
 *                        every row; the caller takes np.percentile(err, 90) as the outlier threshold (:212).
 *   pcm_pca_residuals_k  the same for components[n_components][F] (row-major, 1 <= n_components <=
 *                        PCM_MAX_PCA_COMPONENTS): t_j = x.c_j - mean.c_j, err = sum_f |x_f - (mean_f + sum_j t_j c_jf)|.
 *                        With n_components = 1 it returns the bits of pcm_pca_residuals. */
int pcm_pca_moments(pcm_handle* h, long long rows_id, double* gram, double* sums, int64_t* n_class1);
int pcm_pca_residuals(pcm_handle* h, long long rows_id, const double* mean, const double* component, double* err);
int pcm_pca_residuals_k(pcm_handle* h, long long rows_id, const double* mean, const double* components, int n_components,
                        double* err);

/* ---- parity taps (tests, smoke; not needed by the reference flow) -------- */

/* cv.cvtColor(img, BGR2HSV / BGR2LAB) of an h x w x 3 host image with the same
 * device code the fused kernel uses; space = PCM_SPACE_HSV / PCM_SPACE_LAB. */
int pcm_convert(pcm_handle* h, const uint8_t* bgr, int height, int width, int64_t stride,
                int space, uint8_t* out, int64_t out_stride);

/* Raw star-neighbourhood features of a crop as the reference's getFeatures
 * builds them (:249-277): X[h*w, F] int16 with -1 outside the crop. */
int pcm_gather_features(pcm_handle* h, const uint8_t* frame, int frame_h, int frame_w, int64_t frame_stride,
                        const int rect[4], int16_t* X);

/* Bit 0: keep the per-stage buffers that only the parity taps need -- the float64 P(fg) map (and the novelty map) the
 * score kernel otherwise does not store, and the 0/255 map before dilation.  Bit 1 (test hook): every label takes the
 * exact sequential-float32 path of the decision kernel, not only the labels inside the guard band.  Off by default. */
int pcm_set_debug(pcm_handle* h, int on);

/* Stage dumps of the LAST pcm_update / pcm_update_device on this handle
 * (any pointer may be NULL):
 *   p1[h*w]       blended P(foreground) (:80-95), float64
 *   sa[h*w]       blended novelty error (:57-63, :88-93), float64 (zeros if off)
 *   scores[S]     per-label score as the reference's float32 (:241)
 *   areas[S]      per-label pixel counts (:97)
 *   pre[h*w]      0/255 map before dilation (:242-246); needs pcm_set_debug(h, 1)
 *   n_exact       number of labels decided by the exact sequential-f32 path */
int pcm_debug_last(pcm_handle* h, double* p1, double* sa, float* scores, int64_t* areas,
                   uint8_t* pre, int32_t* n_exact);

/* The colour-conversion lookup tables built at pcm_create (parity of the table
 * construction itself): gamma[256], cbrt[2041] uint16; sdiv[256], hdiv[256] int32. */
int pcm_debug_tables(pcm_handle* h, uint16_t* gamma, uint16_t* cbrt_tab, int32_t* sdiv, int32_t* hdiv);

/* Number of kernel launches issued through this handle so far. */
int64_t pcm_launch_count(const pcm_handle* h);

/* Bytes the HOST-buffer entry points (pcm_update, pcm_iou, pcm_quickshift) have copied so far:
 * out[0] host->device, out[1] device->host.  Label chunks that were not re-sent do not count. */
int pcm_transfer_bytes(const pcm_handle* h, int64_t out[2]);

/* Per-kernel device timing (CUDA events on the handle's stream around every
 * launch while enabled).  Kernel ids: 0 score (fused star features + forests),
 * 1 (retired: the per-label reduction is K1's epilogue), 2 segment_decide, 3 (retired: the exact
 * re-evaluation is part of segment_decide), 4 mask_dilate, 5 iou,
 * 6 planes (colour conversion to planar tiles), 7 novelty (reconstruction error of PCAs with
 * two or more components; launched only for frames that use one).
 * pcm_profile_read synchronises the stream, adds the finished launches to the
 * running totals and returns them (ms_sum[i], count[i] for i < n <= PCM_NUM_KERNELS);
 * reset != 0 clears the totals afterwards. */
#define PCM_NUM_KERNELS 8
int pcm_profile_enable(pcm_handle* h, int on);
int pcm_profile_read(pcm_handle* h, double* ms_sum, int64_t* count, int n, int reset);

#ifdef __cplusplus
}
#endif
#endif /* PCM_B200_H */
