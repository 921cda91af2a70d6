/*
 * og_decoder.h — C ABI of the B200-native OffsetGuided post-network decoder.
 *
 * Drop-in boundary for the reference's decoding path (paths relative to the
 * reference repository hellojialee/OffsetGuided):
 *
 *     decoder/factory.py:52-96   PostProcess.generate_poses        (orchestration)
 *     decoder/factory.py:98-146  PostProcess.flip_augment          (flip-test fusion)
 *     decoder/heatmap.py:15-59   hmp_NMS / topK_channel / joint_dets
 *     decoder/offset.py:8-43     scored_offset
 *     decoder/collect.py:62-236  LimbsCollect.generate_limbs
 *     decoder/group.py:39-240    GreedyGroup.group_skeletons
 *
 * Conventions
 *   - plain C types only: device / host pointers, sizes, an opaque handle and a
 *     CUDA stream passed as void* (cudaStream_t); no C++ exceptions cross the ABI;
 *   - every function returns an og_status (0 = OG_OK); og_last_error() gives the
 *     text of the last failure on the calling thread;
 *   - all maps are float32, NCHW, contiguous (og_decode_features_dev_ex also takes
 *     bfloat16 / float16 maps and image-strided views, og_decode_features_dev_strided
 *     channels-last ones as well); "dev" pointers are device
 *     memory of the handle's GPU, "host" pointers are host memory (pinned memory makes
 *     the copies asynchronous and lets the offset maps stay on the host);
 *   - `stream` is the caller's stream: inputs are consumed in its order.  A handle owns one
 *     stream per result slot (the decode chain of a call) and one for host-input copies;
 *     og_fetch_result / og_fetch_poses is the synchronisation point, and inputs must stay
 *     valid until it returns.  Calls on one handle may come from different caller streams:
 *     every call has its own scratch and result slot;
 *   - a handle is bound to one GPU and one configuration and is not thread-safe;
 *     distinct handles are independent (the image-sharding driver keeps one per GPU);
 *   - there is no CPU fallback: every entry point launches sm_100a kernels.
 *
 * The reference is a Python package, so the binding a maintainer adds is a ctypes
 * stub (INTEGRATION.md); offsetguided_b200/_lib.py is that stub.
 */
#ifndef OG_DECODER_H_
#define OG_DECODER_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OG_ABI_VERSION 2
#define OG_MAX_IN_FLIGHT 16  /* decode calls a handle keeps in flight (result slots) */
#define OG_LIMB_COLS 13      /* decoder/collect.py:220-222 */
#define OG_POSE_COLS 6       /* decoder/group.py:48  [x, y, v, s, limb_score, ind] */
#define OG_MAX_KEYPOINTS 64
#define OG_MAX_LIMBS 64
#define OG_MAX_TOPK 128
#define OG_DTYPE_F32 0       /* element types of og_decode_features_dev_ex */
#define OG_DTYPE_BF16 1
#define OG_DTYPE_F16 2       /* what the reference's apex AMP evaluation produces (evaluate.py:139-150) */

typedef enum og_status {
    OG_OK = 0,
    OG_ERR_INVALID_ARGUMENT = 1,
    OG_ERR_CUDA = 2,
    OG_ERR_OUT_OF_MEMORY = 3,
    OG_ERR_CAPACITY = 4,          /* caller-provided output buffer too small */
    OG_ERR_UNSUPPORTED = 5
} og_status;

/* Configuration = constructor arguments of LimbsCollect (decoder/collect.py:37-60)
 * and GreedyGroup (decoder/group.py:29-37) plus the skeleton table
 * (config/coco_data.py:12-15). */
typedef struct og_config {
    int32_t n_keypoints;          /* C */
    int32_t n_limbs;              /* L */
    const int32_t *limb_from;     /* [L] from-joint of every limb, skeleton order  */
    const int32_t *limb_to;       /* [L] to-joint                                  */
    int32_t topk;                 /* K  (--topk)                                   */
    float thre_hmp;               /* --thre-hmp; score < thre -> moved off image   */
    float min_len;                /* --min-len                                      */
    float resize_factor;          /* off_stride / hmp_stride (collect.py:48)        */
    float dist_max;               /* --dist-max                                     */
    int32_t use_scale;            /* --use-scale: gate is max(dist_max, scale_t)    */
    double person_thre;           /* --person-thre (compared in float64)            */
    int32_t sort_dim;             /* --sort-dim: pose column the person score uses  */
    int32_t device;               /* CUDA device ordinal, -1 = current              */
    int32_t max_images;           /* initial capacity in images (grows on demand)   */
} og_config;

typedef struct og_handle og_handle;

const char *og_last_error(void);
const char *og_status_string(int status);
int og_abi_version(void);

int og_create(const og_config *cfg, og_handle **out);
int og_destroy(og_handle *h);

/* ---- decoder/heatmap.py -------------------------------------------------- */

/* hmp_NMS (heatmap.py:15-35): out = heat * (maxpool3x3_zero_pad(heat) == heat). */
int og_hmp_nms_f32(const float *heat_dev, float *out_dev,
                   int n, int c, int h, int w, void *stream);

/* topK_channel (heatmap.py:38-49): exact per-(n, c) top-K of an arbitrary score
 * map, ordered (value desc, flat index asc).  out_* are [n, c, k]. */
int og_topk_channel_f32(og_handle *h, const float *scores_dev,
                        int n, int c, int hgt, int w, int k,
                        float *out_score_dev, int32_t *out_index_dev, void *stream);

/* joint_dets with the candidate threshold applied first (K1): fused 3x3 NMS +
 * `value >= thre` + per-channel top-K.  Streams the heat map from HBM once.
 * Slots beyond the number of surviving peaks hold score 0 / index -1;
 * out_count_dev[n, c] = number of real candidates (<= k).
 * With thre = -INFINITY this is exactly joint_dets (heatmap.py:52-59). */
int og_nms_topk_f32(og_handle *h, const float *heat_dev,
                    int n, int hgt, int w, float thre,
                    float *out_score_dev, int32_t *out_index_dev,
                    int32_t *out_count_dev, void *stream);

/* ---- decoder/collect.py -------------------------------------------------- */

/* generate_limbs from the candidate tables (K2, collect.py:100-233).
 * offs_dev [n, 2L, h, w]; scales_dev [n, C, h, w] or NULL (scale = 4, collect.py:117).
 * out_limbs_dev [n, L, K, 13]. */
int og_limb_score_f32(og_handle *h, const float *det_score_dev, const int32_t *det_index_dev,
                      const float *offs_dev, const float *scales_dev,
                      int n, int hgt, int w, float *out_limbs_dev, void *stream);

/* generate_limbs with the optional heads (collect.py:127-138, 158-165, 213-218):
 * jomps_dev [n, 2, h, w] jitter-offset maps or NULL, use_jitter = --use-jitter-offset,
 * vector_nd = 4 for the cat_flip_offs offsets ([n, 4L, h, w], factory.py:115-127). */
int og_limb_score_ex_f32(og_handle *h, const float *det_score_dev, const int32_t *det_index_dev,
                         const float *offs_dev, const float *scales_dev, const float *jomps_dev,
                         int vector_nd, int use_jitter, int n, int hgt, int w, float *out_limbs_dev,
                         void *stream);

/* ---- decoder/group.py ---------------------------------------------------- */

/* group_skeletons for n images (K3, one CTA per image).  limbs_dev [n, L, K, 13].
 * Poses are packed into out_poses_dev [capacity_rows, C, 6]; image i owns rows
 * [out_offset_dev[i], out_offset_dev[i] + out_count_dev[i]).  out_total_dev[0] is
 * the number of rows all images produced; rows beyond capacity_rows are dropped
 * (compare out_total with capacity_rows). */
int og_group_f32(og_handle *h, const float *limbs_dev, int n,
                 float *out_poses_dev, int32_t capacity_rows,
                 int32_t *out_offset_dev, int32_t *out_count_dev, int32_t *out_total_dev,
                 void *stream);

/* ---- decoder/offset.py, decoder/factory.py ------------------------------- */

/* scored_offset (offset.py:8-43) with a k x k window, out_dev [n, 2L, h, w]. */
int og_scored_offset_f32(og_handle *h, const float *hmp_dev, const float *off_dev,
                         int n, int hgt, int w, int kernel_size, float *out_dev, void *stream);

/* flip_augment, vector-addition branch (factory.py:98-106, 128-139).
 * Inputs hold n originals followed by n W-flipped copies. */
int og_flip_fuse_f32(og_handle *h, const float *hmp2n_dev, const float *off2n_dev,
                     const int32_t *kp_flip, const int32_t *limb_flip,
                     const int32_t *limb_reserve, int n_reserve,
                     int n, int hgt, int w, float *out_hmp_dev, float *out_off_dev, void *stream);

/* Flip fusion of a generic map stack (heat, scale, jitter maps; factory.py:101-113, 141-144):
 * out[i, c] = (in[i, c] + sign * flip_W(in[n + i, perm[c]])) / 2, perm = NULL for identity,
 * sign = -1 on even channels when negate_even (x components of jitter maps). */
int og_flip_average_f32(const float *in2n_dev, const int32_t *perm, int negate_even, int n, int ch,
                        int hgt, int w, float *out_dev, void *stream);

/* flip_augment, cat_flip_offs branch (factory.py:115-127): out_dev [n, 4L, h, w] holds
 * (x, y, x_flip, y_flip) per limb; reserved limbs repeat their original vector. */
int og_flip_cat_offsets_f32(const float *off2n_dev, const int32_t *limb_flip,
                            const int32_t *limb_reserve, int n_reserve, int n, int n_limbs, int hgt,
                            int w, float *out_dev, void *stream);

/* F.interpolate(scale_factor=scale, align_corners=False) (factory.py:74-78);
 * mode 0 = bilinear, 1 = bicubic (A = -0.75). in [planes, h, w] -> out [planes, h*s, w*s]. */
int og_resize_f32(const float *in_dev, float *out_dev, int planes, int hgt, int w,
                  int scale, int mode, void *stream);

/* ---- whole path ----------------------------------------------------------- */

/* generate_limbs + group_skeletons on full-resolution device maps: K1 on `stream`
 * (after whatever produced the maps there), then K2 -> K3 on a high-priority stream OWNED BY
 * THE HANDLE (one per result slot), ordered after K1 by an event; K3 writes the packed poses
 * straight into pinned host memory of the handle.  K2 / K3 are latency-bound and fill a
 * fraction of the SMs, so the next call's K1 (HBM-bound) runs beside them instead of behind them.
 * Returns immediately; og_fetch_result() synchronises.  Every input buffer of an og_decode_*
 * call must stay valid and unmodified until its og_fetch_poses returns (K2 reads the offset
 * maps after the call has returned, not in `stream` order). */
int og_decode_maps(og_handle *h, const float *heat_dev, const float *offs_dev,
                   const float *scales_dev, int n, int hgt, int w, void *stream);

/* og_decode_maps with the optional heads of og_limb_score_ex_f32. */
int og_decode_maps_ex(og_handle *h, const float *heat_dev, const float *offs_dev,
                      const float *scales_dev, const float *jomps_dev, int vector_nd, int use_jitter,
                      int n, int hgt, int w, void *stream);

/* PostProcess.generate_poses on NETWORK-RESOLUTION maps held in HOST memory:
 * H2D copy, optional flip fusion (hmp_host has 2n images then), x stride resize
 * (mode as og_resize_f32), K1 -> K2 -> K3, D2H of the poses.
 * kp_flip / limb_flip / limb_reserve may be NULL when flip_test == 0. */
int og_decode_features_host(og_handle *h, const float *hmp_host, const float *off_host,
                            int n, int hgt, int w, int hmp_stride, int off_stride,
                            int resize_mode, int flip_test,
                            const int32_t *kp_flip, const int32_t *limb_flip,
                            const int32_t *limb_reserve, int n_reserve, void *stream);

/* Same on device-resident network-resolution maps (what evaluate.py:215 hands over).
 * `stream` is only waited on: the whole chain (fused flip + resize + NMS, selection, limb
 * scoring, grouping) runs on the result slot's own stream, as ONE CUDA graph captured per slot
 * and replayed while the input pointers, shapes, flags and flip tables stay the same (the
 * usual case: a network writes its outputs to the same buffers every iteration); anything
 * else re-captures.  og_set_graph(h, 0) launches the kernels one by one instead. */
int og_decode_features_dev(og_handle *h, const float *hmp_dev, const float *off_dev,
                           int n, int hgt, int w, int hmp_stride, int off_stride,
                           int resize_mode, int flip_test,
                           const int32_t *kp_flip, const int32_t *limb_flip,
                           const int32_t *limb_reserve, int n_reserve, void *stream);

/* og_decode_features_dev on maps as a reduced-precision network leaves them (SURVEY 8f-4; the
 * reference converts everything to float32 first, decoder/factory.py:59): `dtype` OG_DTYPE_F32,
 * OG_DTYPE_BF16 or OG_DTYPE_F16; consecutive images are `hmp_image_stride` / `off_image_stride` ELEMENTS apart
 * (0 = dense), the C (resp. 2L) planes of one image are contiguous — so the two channel slices
 * of one packed [n, C + 2L, h, w] head output are decoded in place, without a split or a
 * float32 copy.  bf16 / f16 values widen exactly to float32: results are bit-identical to
 * decoding the converted maps.  Fused path only (strides 2 / 4 / 8, thre_hmp > 0); the exact redo of a
 * candidate overflow converts the maps to dense float32 on the device first.  Equivalent to
 * og_decode_features_dev_strided with planar strides. */
int og_decode_features_dev_ex(og_handle *h, const void *hmp_dev, const void *off_dev, int dtype,
                              int64_t hmp_image_stride, int64_t off_image_stride,
                              int n, int hgt, int w, int hmp_stride, int off_stride,
                              int resize_mode, int flip_test,
                              const int32_t *kp_flip, const int32_t *limb_flip,
                              const int32_t *limb_reserve, int n_reserve, void *stream);

/* og_decode_features_dev_ex for maps in either memory layout, such as the outputs of a network run
 * in PyTorch's channels_last format, decoded in place without a transposing copy.  Each map is
 * described by its element strides in (image, channel, row, column) order, as Tensor.stride()
 * reports them; the two maps are classified independently:
 *   planar         (s_n, hgt * w, w, 1), s_n >= channels * hgt * w;
 *   channels-last  (s_n, 1, w * p, p), p >= channels (p = channel count of the whole packed tensor,
 *                  the base pointer may sit at any element), s_n >= hgt * w * p.
 * s_n is not checked when the buffer holds one image; a layout that is both is planar.  Any other
 * strides return OG_ERR_INVALID_ARGUMENT before anything is launched.  Channels-last heat maps are
 * read once by a transposing scan that writes them, flip-fused, as dense float32 planes into a
 * scratch buffer of the result slot (n * C * hgt * w * 4 bytes, allocated by the first such call);
 * results are bit-identical to decoding contiguous float32 copies.  Fused path only, like
 * og_decode_features_dev_ex. */
int og_decode_features_dev_strided(og_handle *h, const void *hmp_dev, const void *off_dev, int dtype,
                                   const int64_t hmp_elem_strides[4], const int64_t off_elem_strides[4],
                                   int n, int hgt, int w, int hmp_stride, int off_stride,
                                   int resize_mode, int flip_test,
                                   const int32_t *kp_flip, const int32_t *limb_flip,
                                   const int32_t *limb_reserve, int n_reserve, void *stream);

/* og_decode_features_dev with the optional heads and flags of PostProcess.generate_poses
 * (decoder/factory.py:52-96, collect.py:111-138, 158-165, 213-218), still on the fused path: the
 * keypoint-scale maps `scale_dev` [n or 2n, C, hgt, w] (--include-scale; resized like the heat maps
 * in the reference) and the jitter-offset maps `jitter_dev` [n or 2n, 2, hgt, w]
 * (--include-jitter-offset; bilinear) are interpolated by K2 at the candidate pixels only, with
 * their flip-test averages (factory.py:109-113, 141-144) fused in; `cat_flip_offs` scores the limbs
 * on the 4-D vectors [original, mirrored copy] (factory.py:115-127) instead of their average.
 * Either map pointer may be NULL.  Dense float32 maps; same results, bit for bit, as
 * materialising every map and calling og_decode_maps_ex. */
int og_decode_features_heads_dev(og_handle *h, const float *hmp_dev, const float *off_dev,
                                 const float *scale_dev, const float *jitter_dev, int n, int hgt, int w,
                                 int hmp_stride, int off_stride, int resize_mode, int flip_test,
                                 int cat_flip_offs, int use_jitter, const int32_t *kp_flip,
                                 const int32_t *limb_flip, const int32_t *limb_reserve, int n_reserve,
                                 void *stream);

/* A prepared og_decode_features_dev_ex: a network writes its outputs to the same buffers batch
 * after batch, so a caller validates and records the arguments once (og_plan_features, which
 * also installs the flip tables) and then launches each batch with three arguments.  A plan stays
 * valid for the life of the handle while the buffers exist and the flip tables are unchanged.
 * The strides are validated when the plan is made. */
int og_plan_features(og_handle *h, const void *hmp_dev, const void *off_dev, int dtype,
                     int64_t hmp_image_stride, int64_t off_image_stride, int n, int hgt, int w,
                     int hmp_stride, int off_stride, int resize_mode, int flip_test,
                     const int32_t *kp_flip, const int32_t *limb_flip, const int32_t *limb_reserve,
                     int n_reserve, int32_t *plan_id);
/* og_plan_features for og_decode_features_dev_strided: planar or channels-last maps. */
int og_plan_features_strided(og_handle *h, const void *hmp_dev, const void *off_dev, int dtype,
                             const int64_t hmp_elem_strides[4], const int64_t off_elem_strides[4],
                             int n, int hgt, int w, int hmp_stride, int off_stride, int resize_mode,
                             int flip_test, const int32_t *kp_flip, const int32_t *limb_flip,
                             const int32_t *limb_reserve, int n_reserve, int32_t *plan_id);
int og_plan_launch(og_handle *h, int32_t plan_id, void *stream);

/* Up to OG_MAX_IN_FLIGHT og_decode_* calls may be in flight on a handle (results are queued in
 * order): every call owns a result slot with its own stream, scratch and pinned result buffer,
 * so the kernels of consecutive calls overlap each other and the host-side consumption of
 * batch i (two in flight hide the host round trip when K1 is long; with 8-image shards of a
 * batch split over several GPUs a call is ~0.05 ms of latency-bound kernels and only several
 * calls in flight keep a GPU busy).
 * og_fetch_result waits for the OLDEST unfetched call and exposes its result: `poses` points
 * into pinned memory owned by the handle ([total_rows, C, 6] float32, written there by the
 * grouping kernel itself), image i owns rows [offsets[i], offsets[i] + counts[i]); the
 * pointers stay valid until OG_MAX_IN_FLIGHT further og_decode_* calls have been made.
 * og_fetch_poses is the same without the image count; og_pending returns the number of
 * unfetched calls. */
typedef struct og_result {
    const float *poses;          /* [total_rows, n_keypoints, 6] */
    const int32_t *offsets;      /* [n_images] first row of every image */
    const int32_t *counts;       /* [n_images] persons of every image   */
    int32_t n_images;            /* images of the decode call this result belongs to */
    int32_t total_rows;
    int32_t n_keypoints;
    int32_t buffer_id;           /* changes whenever the pointers refer to another (re-allocated) buffer */
    /* only after og_set_frames (else NULL): the result rows of the reference's evaluation loop,
     * row r of these arrays = pose row r */
    const float *coco_keypoints; /* [total_rows, 3 * n_keypoints]  x, y, flag per keypoint */
    const double *coco_scores;   /* [total_rows]  mean keypoint score                      */
    const int32_t *coco_images;  /* [total_rows]  image index within the call              */
} og_result;
int og_fetch_result(og_handle *h, og_result *out);

/* Pose back-projection and result rows on the GPU (replaces the per-image / per-person /
 * per-keypoint Python loops of transforms/preprocess.py:33-63 annotations_inverse and
 * evaluate.py:227-265).  og_set_frames stages, for the NEXT og_decode_* call on the handle, the
 * frame of each of its n images: frames_host[4 i ..] = { offset_x, offset_y, scale_x, scale_y }
 * (meta['offset'], meta['scale']).  The grouping kernel then also writes, for every person,
 * x' = around((x + offset_x) / scale_x, 2), y' likewise, flag = (x' > 0 or y' > 0) per keypoint
 * and score = sum(v) / C, with the reference's rounding (float64 steps rounded to float32, numpy's
 * float32 around, float64 score); og_fetch_result exposes them next to the poses. */
int og_set_frames(og_handle *h, const double *frames_host, int n);
int og_fetch_poses(og_handle *h, const float **poses_host, const int32_t **offset_host,
                   const int32_t **count_host, int32_t *total_rows);
int og_pending(const og_handle *h);

/* Copy the device-side intermediates of the last decode call (n images) into
 * caller-provided device buffers (any may be NULL): det scores [n, C, K],
 * det indices [n, C, K], limbs [n, L, K, 13].  For tests and debugging. */
int og_copy_intermediates(og_handle *h, int n, float *det_score_dev, int32_t *det_index_dev,
                          float *limbs_dev, void *stream);

/* Number of kernels this library has launched through the handle so far. */
int64_t og_launch_count(const og_handle *h);

/* og_decode_features_* use a fused path by default (strides 2/4/8, thre_hmp > 0): flip
 * fusion + resize + NMS in one kernel over the network-resolution maps, offsets sampled at
 * the candidates; results are bit-identical to the materialising path.  If a heat-map plane
 * yields more than 2048 candidates (noise-like input), og_fetch_result materialises that plane
 * alone at full resolution, selects its top-K exactly and runs the limb scoring and grouping of
 * the batch again on the completed detections; the input buffers of og_decode_features_dev must
 * therefore stay valid until the result has been fetched.  og_set_fused(h, 0) disables the fused
 * path; og_fused_redo_count reports how many batches needed such a redo. */
int og_set_fused(og_handle *h, int enable);

/* Device path of og_decode_features_dev[_ex]: replay a captured CUDA graph per result slot
 * (default) or launch kernel by kernel; the counters report replays and (re)captures. */
int og_set_graph(og_handle *h, int enable);
int64_t og_graph_replay_count(const og_handle *h);
int64_t og_graph_build_count(const og_handle *h);

/* Development aid: per-phase clock64() totals of the K3 CTA kernel; only in builds with
 * -DOG_K3_PROFILE (returns OG_ERR_UNSUPPORTED otherwise). */
int og_debug_k3_profile(uint64_t *out16, int reset);
int64_t og_fused_redo_count(const og_handle *h);
/* K3 groups an image with one warp and a 64-row person table in shared memory.  An image that
 * needs more rows (noise-like input) is grouped by the CTA kernel (tables in global memory)
 * when its batch is fetched; og_k3_redo_count reports how many fetches did that. */
int64_t og_k3_redo_count(const og_handle *h);

/* og_decode_features_host, fused path: when `off_host` is pinned (device-accessible) host memory
 * the offset maps are NOT copied to the device — K2 reads its 2 * L * K bilinear samples per image
 * straight from the host buffer over PCIe (a few KB instead of 2L * h * w * 4 bytes per image).
 * Pageable buffers are copied as a whole.  The host buffers must stay valid and unmodified until
 * og_fetch_poses returns (this already holds for the asynchronous copies).  og_set_zero_copy(h, 0)
 * forces the full copy; og_zero_copy_count reports how many calls left the offsets on the host.
 * (replaces the reference's implicit "everything lives on the model's device",
 * decoder/factory.py:59-63) */
int og_set_zero_copy(og_handle *h, int enable);
int64_t og_zero_copy_count(const og_handle *h);

/* Per-stage device timing of og_decode_* calls with CUDA events recorded on the stream
 * each stage is launched on (while it is enabled the device path launches kernel by kernel
 * instead of replaying its graph).  og_last_stage_times_ms() reports the most recently FETCHED
 * decode call: out6 = { input copy + flip + resize, K1 pass 1 (NMS stream / fused scan + list +
 * blocks), K1 pass 2 (select), K2 (+ row preparation), K3, end-of-chain marker (the poses are
 * written to host memory by K3 itself: ~0) } in milliseconds. */
int og_enable_stage_timing(og_handle *h, int enable);
int og_last_stage_times_ms(og_handle *h, float *out6);

#ifdef __cplusplus
}
#endif
#endif  /* OG_DECODER_H_ */
