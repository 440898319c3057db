/*
 * spgroup.h -- C ABI of the B200-native keypoint-grouping path (libspgroup.so).
 *
 * Drop-in boundary for SimplePose's post-network grouping stage.  The reference
 * (hellojialee/Improved-Body-Parts) has no plugin/FFI layer: the boundary is three module-level
 * Python functions called back to back at /root/reference/evaluate.py:509-511 plus two helpers in
 * utils/util.py.  Each entry point below names the reference interface it replaces; INTEGRATION.md
 * shows the ctypes binding a maintainer adds to evaluate.py.
 *
 * Conventions
 *   - plain C: opaque handle, POD structs, raw pointers and sizes; no torch / C++ types.
 *   - every function returns 0 (SPG_OK) or a negative SPG_E_* code; spg_last_error() gives a message.
 *   - device pointers are raw CUDA device addresses in the handle's device's primary context;
 *     `stream` is a cudaStream_t passed as void* (NULL = default stream).  Kernel launches are
 *     asynchronous on that stream; the *_download_* / spg_group_host calls synchronise it.
 *   - maps are channel-first float planes with contiguous rows (pixel stride 1, row stride W);
 *     image and channel strides are given in ELEMENTS.  The network's raw [N,50,h,w] tensor can be
 *     passed directly with channel offsets 0 (body parts) / 30 (keypoints), config/config.py:101-103.
 *   - no CPU fallback exists: without a usable sm_100 device spg_create fails.
 *   - per-image problems (capacity overflows, an out-of-range sample index where the reference would
 *     raise IndexError) are reported in the status word of that image, never by exceptions.
 */
#ifndef SPGROUP_H_
#define SPGROUP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPG_ABI_VERSION 2

enum {
    SPG_OK = 0,
    SPG_E_INVALID = -1,   /* bad argument (shape, capacity, alignment, null pointer) */
    SPG_E_CUDA = -2,      /* a CUDA runtime call failed; see spg_last_error          */
    SPG_E_NO_DEVICE = -3, /* no CUDA device / not an sm_100 part                     */
    SPG_E_STATE = -4      /* stage called before the stage that feeds it             */
};

/* per-image status bits (spg_download_status) */
enum {
    SPG_ST_PEAK_OVERFLOW = 1u << 0,  /* a part class had more peaks than max_peaks_per_part      */
    SPG_ST_CAND_OVERFLOW = 1u << 1,  /* a limb had more surviving candidates than max_cands      */
    SPG_ST_ROW_OVERFLOW = 1u << 2,   /* person assembly needed more than max_person_rows rows    */
    SPG_ST_SAMPLE_INDEX = 1u << 3,   /* a line sample fell outside the map: the reference would  */
                                     /* raise IndexError at evaluate.py:235                      */
    SPG_ST_ASSERT = 1u << 4,         /* the reference would raise at evaluate.py:437-439         */
    SPG_ST_WIRE_OVERFLOW = 1u << 5   /* more persons than the wire record holds (rows beyond are dropped) */
};

/* dtype of the body-part planes.  predict() accumulates them in float64 (evaluate.py:86,161); with a single scale
 * (the reference's default, utils/config:26) every float64 value is exactly a float32 one, so the planes can be STORED
 * as float32 and evaluated with the float64 arithmetic the reference applies: SPG_F32_AS_F64 -- half the HBM traffic,
 * bit-identical results to SPG_F64 planes holding the same values.  SPG_F16 is accepted for network outputs only. */
enum { SPG_F32 = 0, SPG_F64 = 1, SPG_F32_AS_F64 = 2, SPG_F16 = 3 };

typedef struct spg_handle spg_handle;

/* Skeleton + capacities.  Mirrors config/config.py:52-126 (runtime data, not compile-time). */
typedef struct spg_config {
    int32_t abi_version;        /* SPG_ABI_VERSION */
    int32_t device;             /* CUDA device ordinal */
    int32_t n_parts;            /* K: keypoint channels used (18; evaluate.py:175,187) */
    int32_t n_limbs;            /* L: body-part channels (30; config.py:94-96) */
    const int32_t *limbs;       /* [L][2] (from_part, to_part) = limbs_conn */
    int32_t n_out_joints;       /* 17 COCO joints */
    const int32_t *out_from_part; /* [n_out_joints] part index feeding each output joint (inverse of dt_gt_mapping, config.py:117) */
    int32_t max_batch;          /* images resident per call */
    int32_t max_h, max_w;       /* largest map */
    int32_t max_peaks_per_part; /* <= 128 */
    int32_t max_cands_per_limb; /* surviving candidates kept per (image, limb) */
    int32_t max_person_rows;    /* <= 128; rows of `subset` alive or dead during assembly */
} spg_config;

/* Grouping hyper-parameters: the reference's `params` dict (utils/config:17-28) plus the two literals of
 * the final prune (evaluate.py:493). */
typedef struct spg_params {
    double thre1, thre2, connect_ration, len_rate, connection_tole, min_mean_score;
    int32_t mid_num, offset_radius, remove_recon, min_parts;
    /* demo_image.py's inlined copy of the grouping code differs from evaluate.py in two decisions (SURVEY 3.2); both 0
     * for evaluate.py.  With min_parts = 4 (demo_image.py:533) they give the demo's behaviour. */
    int32_t crit1_strict;       /* 1: `count >  connect_ration*n` (demo_image.py:288) instead of `>=` (evaluate.py:246) */
    int32_t refresh_len_check;  /* 1: the same-B refresh also requires len_rate*maxlen > len (demo_image.py:414-415)   */
} spg_params;

/* Device-resident results of the last call, for consumers that stay on the GPU (NCCL gather, benchmarks).
 * All arrays are indexed [image][...] with the capacities of spg_config. */
typedef struct spg_device_view {
    int32_t max_batch, n_parts, n_limbs, n_out_joints, cap_peaks, cap_cands, cap_rows;
    /* peaks: [N][K][cap_peaks] */
    const double *peak_x, *peak_y;     /* refined coordinates (util.py:204-211) */
    const float *peak_score;
    const uint32_t *peak_anchor;       /* (y << 16) | x integer anchor; bit 31 = border peak (integer coords, util.py:201-202) */
    const int32_t *peak_count;         /* [N][K] true count (may exceed cap -> status bit) */
    /* connections: [N][L][cap_peaks] in greedy acceptance order (evaluate.py:263-270) */
    const uint32_t *conn_ij;           /* (i << 16) | j */
    const double *conn_score, *conn_norm;
    const int32_t *conn_count;         /* [N][L]; -1 = special_k (evaluate.py:272-274) */
    const int32_t *cand_count;         /* [N][L] candidates that passed both criteria (evaluate.py:252) */
    const int32_t *surv_count;         /* [N][L] pairs that survived the scoring kernel's conservative screen (diagnostic) */
    /* persons */
    const double *subset;              /* [N][cap_rows][K+2][2] after the prune (evaluate.py:491-496) */
    const int32_t *n_persons;          /* [N] */
    const double *people_xy;           /* [N][cap_rows][n_out_joints][2] (evaluate.py:523-539) */
    const double *people_score;        /* [N][cap_rows]  1 - 1/total (evaluate.py:541) */
    const uint32_t *status;            /* [N] SPG_ST_* bits */
} spg_device_view;

/* ---- lifetime -------------------------------------------------------------------------------- */
int spg_create(const spg_config *cfg, spg_handle **out);
void spg_destroy(spg_handle *h);
const char *spg_last_error(const spg_handle *h); /* h may be NULL: last creation error */
int spg_abi_version(void);
int spg_get_device_view(const spg_handle *h, spg_device_view *out);

/* ---- whole path: replaces the three calls at evaluate.py:509-511 ------------------------------ */
/* device inputs already resident; asynchronous on `stream` */
int spg_group_batch(spg_handle *h, const float *heat_dev, int64_t heat_image_stride, int64_t heat_chan_stride,
                    const void *paf_dev, int32_t paf_dtype, int64_t paf_image_stride, int64_t paf_chan_stride,
                    int32_t n_images, int32_t height, int32_t width, double image_extent,
                    const spg_params *params, void *stream);

/* host inputs (pinned for full overlap; pageable works): H2D in chunks overlapped with the kernels, results
 * copied back into the caller's arrays (any of which may be NULL).  Synchronous.
 *   heat_host [N][K][H][W] f32, paf_host [N][L][H][W] f32|f64
 *   out_n_persons [N], out_people_xy [N][cap_rows][J][2], out_people_score [N][cap_rows], out_status [N] */
int spg_group_host(spg_handle *h, const float *heat_host, const void *paf_host, int32_t paf_dtype,
                   int32_t n_images, int32_t height, int32_t width, double image_extent,
                   const spg_params *params, int32_t *out_n_persons, double *out_people_xy,
                   double *out_people_score, uint32_t *out_status);

/* pinned host memory for spg_group_host callers that do not have their own */
int spg_host_alloc(void **ptr, uint64_t bytes);
int spg_host_free(void *ptr);

/* ---- post-network stage: the scale loop of predict() after the forward pass, evaluate.py:126-161 ----------- */
/* One entry per (scale) of params['scale_search']: the network's output for a batch of image pairs
 * [N][2][C][h][w] (image, mirrored image; evaluate.py:116-126), device memory, float32 or float16. */
typedef struct spg_postnet_scale {
    const void *net_out;
    int32_t dtype;                  /* SPG_F32 | SPG_F16 */
    int64_t image_stride, pair_stride, chan_stride; /* elements; rows are contiguous (row stride w) */
    int32_t h, w;                   /* network output size = padded input size / stride */
    int32_t crop_h, crop_w;         /* imageToTest size: padded size minus pad[2] / pad[3] (evaluate.py:148) */
} spg_postnet_scale;
typedef struct spg_postnet_desc {
    int32_t n_scales;               /* items of the loop: len(multiplier) * len(rotate_angle) (spg_postnet: angle 0 only) */
    const spg_postnet_scale *scales;
    int32_t stride;                 /* model_params['stride'] (4) */
    int32_t paf_chan0, heat_chan0;  /* first body-part / keypoint channel of the network output (0 / 30, config.py:101-103) */
    const int32_t *flip_paf_ord;    /* [n_limbs]  config.py:121-124 */
    const int32_t *flip_heat_ord;   /* [n_parts] */
    int32_t nan_scrub;              /* demo_image.py:179-180: NaN -> 0 in the averaged maps (evaluate.py: 0) */
} spg_postnet_desc;
/* flip ensemble (:139-140) + cv2.resize x stride (:143,152) + crop (:148,157) + cv2.resize to the image (:149,158) +
 * float64 average over the scales (:160-161), fused, writing the channel-first planes the grouping kernels stream:
 *   heat_out [N][n_parts][H][W] float32 (the cast of evaluate.py:173 applied),
 *   paf_out  [N][n_limbs][H][W] SPG_F64, or SPG_F32 when n_scales == 1 (then pass SPG_F32_AS_F64 to the grouping calls).
 * Interpolation follows OpenCV's generic bicubic path (A = -0.75) operation for operation in float32. */
int spg_postnet(spg_handle *h, const spg_postnet_desc *desc, int32_t n_images, int32_t height, int32_t width,
                float *heat_out, void *paf_out, int32_t paf_dtype, void *stream);
/* The same with rotation search (evaluate.py:90-158 with rotation_search != [0]): desc->n_scales counts the items of
 * product(multiplier, rotate_angle) in the loop's order (scale-major, angle-minor), angle_deg[n_scales] their angles in
 * degrees.  For an item with angle != 0 the up-sampled maps are warped back over the whole padded image before the crop
 * -- cv2.warpAffine(map, getRotationMatrix2D((Hp / 2, Wp / 2), -angle, 1), (0, 0)) with Hp = h * stride, Wp = w * stride,
 * the centre's (rows, cols) order as in the reference -- following OpenCV's fixed-point INTER_LINEAR / BORDER_CONSTANT 0
 * path bit for bit.  The caller warps the network input with the matching getRotationMatrix2D(..., angle, 1).  Items with
 * angle 0 take spg_postnet's kernels; all angles 0 is spg_postnet.  Non-finite angles: SPG_E_INVALID.  SPG_F32 body-part
 * planes need n_scales == 1, as for spg_postnet. */
int spg_postnet_rotated(spg_handle *h, const spg_postnet_desc *desc, const double *angle_deg, int32_t n_images,
                        int32_t height, int32_t width, float *heat_out, void *paf_out, int32_t paf_dtype, void *stream);

/* ---- pre-network stage: one scale of predict()'s loop before the forward pass, evaluate.py:98-116 ----------- */
/* Host only, no handle: the sizes spg_prenet produces for a height x width image at `scale` --
 * crop = imageToTest.shape[:2] = (rint(height * scale), rint(width * scale)) (cv2.resize's dsize, round half to even in
 * float64; what spg_postnet crops to) and pad = imageToTest_padded.shape[:2] (crop rounded up to multiples of
 * max_downsample, utils/util.py:44-64).  SPG_E_INVALID for an image outside [1, 32767], a scale that is not finite or
 * <= 0, max_downsample <= 0, an empty crop or a padded size above 32767; spg_last_error(NULL) gives the reason. */
int spg_prenet_size(int32_t height, int32_t width, double scale, int32_t max_downsample, int32_t *crop_h, int32_t *crop_w,
                    int32_t *pad_h, int32_t *pad_w);
/* The network input of every angle of one scale:
 *   cv2.resize(image, (0, 0), fx=scale, fy=scale, INTER_CUBIC) -> padRightDownCorner(max_downsample, pad_value) -> / 255
 *   -> cv2.warpAffine(getRotationMatrix2D((Hp / 2, Wp / 2), angle, 1), (0, 0)) for angle != 0 -> [image, mirrored image]
 * image_dev: uint8 HWC device image, `channels` must be 3, pixels contiguous, `row_stride` bytes between rows (a crop of
 * a larger frame works).  out + k * item_stride (elements) receives angle_deg[k]'s item as float32 [2][Hp][Wp][3], the
 * layout the reference feeds its network.  The resize is OpenCV's 8-bit generic bicubic path without IPP, bit for bit
 * (cv2 with IPP, its default, differs by at most 1 in a few percent of the uint8 values); the warp is warpAffine's
 * fixed-point INTER_LINEAR path with border 0, as spg_postnet_rotated's.  Two launches for the first angle, one per
 * further angle; the padded image lives in handle workspace that grows on demand.  Asynchronous on `stream`.
 * SPG_E_INVALID for channels != 3, pad_value outside [0, 255], a non-finite angle, and spg_prenet_size's cases. */
int spg_prenet(spg_handle *h, const unsigned char *image_dev, int64_t row_stride, int32_t height, int32_t width,
               int32_t channels, double scale, const double *angle_deg, int32_t n_angles, int32_t max_downsample,
               int32_t pad_value, float *out, int64_t item_stride, void *stream);

/* ---- stage entry points (stage-wise parity; each consumes the previous stage's device state) ---- */
/* find_peaks: evaluate.py:169-203 = util.keypoint_heatmap_nms (utils/util.py:177-183) + util.refine_centroid (:186-211) */
int spg_nms_peaks(spg_handle *h, const float *heat_dev, int64_t image_stride, int64_t chan_stride,
                  int32_t n_images, int32_t height, int32_t width, const spg_params *params, void *stream);
/* find_connections, scoring half: evaluate.py:211-255 (every candidate pair of every limb) */
int spg_limb_score(spg_handle *h, const void *paf_dev, int32_t paf_dtype, int64_t image_stride,
                   int64_t chan_stride, int32_t n_images, int32_t height, int32_t width, double image_extent,
                   const spg_params *params, void *stream);
/* find_connections, matching half: evaluate.py:259-274 (stable sort by priority + greedy assignment) */
int spg_limb_match(spg_handle *h, int32_t n_images, const spg_params *params, void *stream);
/* find_people + process() tail: evaluate.py:279-498 and :523-543 */
int spg_assemble(spg_handle *h, int32_t n_images, const spg_params *params, void *stream);
/* the two previous stages fused in one kernel (one CTA per image: matcher warps feed the assembler warp limb by limb
 * through shared memory); what spg_group_batch / spg_group_host run.  Same outputs as the two calls back to back. */
int spg_match_assemble(spg_handle *h, int32_t n_images, const spg_params *params, void *stream);

/* ---- host <-> device state transfer for the stage-wise drop-in functions ---------------------- */
/* peaks of ONE image, part-major flat arrays as the reference's all_peaks flattens (evaluate.py:283):
 * part_count[K], x[n], y[n], score[n] with n = sum(part_count); image_index selects the slot */
int spg_upload_peaks(spg_handle *h, int32_t image_index, const int32_t *part_count, const double *x, const double *y,
                     const float *score, void *stream);
/* connections of ONE image: conn_count[L] (-1 = special), rows concatenated over limbs:
 * ij[m][2] (indices inside candA/candB), score[m], norm[m] */
int spg_upload_connections(spg_handle *h, int32_t image_index, const int32_t *conn_count, const int32_t *ij,
                           const double *score, const double *norm, void *stream);

/* downloads synchronise `stream`.  Arrays are dense with the handle's capacities; NULL pointers are skipped. */
int spg_download_peaks(spg_handle *h, int32_t n_images, int32_t *peak_count /*[N][K]*/, double *x, double *y,
                       float *score, uint32_t *anchor /*[N][K][cap_peaks] each*/, void *stream);
int spg_download_connections(spg_handle *h, int32_t n_images, int32_t *conn_count /*[N][L]*/,
                             int32_t *cand_count /*[N][L]*/, uint32_t *ij, double *score,
                             double *norm /*[N][L][cap_peaks] each*/, void *stream);
int spg_download_people(spg_handle *h, int32_t n_images, int32_t *n_persons /*[N]*/,
                        double *subset /*[N][cap_rows][K+2][2]*/, double *people_xy /*[N][cap_rows][J][2]*/,
                        double *people_score /*[N][cap_rows]*/, void *stream);
int spg_download_status(spg_handle *h, int32_t n_images, uint32_t *status /*[N]*/, void *stream);

/* ---- wire records: what leaves the GPU (format_results, evaluate.py:563-582) ------------------------------- */
/* One fixed-stride record per image: an 8-byte header followed by `rows` person rows of (2*n_out_joints + 2)
 * 8-byte words -- x0,y0,...,x16,y16 (doubles, COCO order, evaluate.py:523-539), the person score 1 - 1/total
 * (double, :541), and a uint64 presence mask (bit g set: joint g was found; clear: the reference's `X, Y = 0, 0`
 * placeholder, :531) -- i.e. exactly the payload format_results turns into {"keypoints": [x,y,v]*17, "score": s}
 * (v = x>0 or y>0).
 * Only the first n_persons rows are written; the rest of the slot is never touched, so when the record lives in
 * another GPU's memory only live rows cross NVLink. */
typedef struct spg_wire_header {
    int32_t n_persons;
    uint32_t status; /* SPG_ST_* bits of the image */
} spg_wire_header;
/* bytes of one image's record for this handle: 8 + wire_rows * (2*n_out_joints + 2) * 8 */
int64_t spg_wire_record_bytes(const spg_handle *h);
/* Direct the assemble stage to ALSO emit wire records: image i of a call goes to
 * (char*)wire_dev + (first_record + i) * spg_wire_record_bytes().  `wire_dev` may be local device memory or PEER
 * memory (another GPU's buffer opened with spg_wire_open: the records then travel over NVLink as the kernel stores
 * them -- the gather of the person lists fused into the kernel that produces them, no collective kernel).
 * wire_rows <= max_person_rows caps the rows per record (SPG_ST_WIRE_OVERFLOW).  NULL switches wire output off. */
int spg_set_wire_output(spg_handle *h, void *wire_dev, int64_t first_record, int32_t wire_rows);

/* Arm the NEXT single-launch assemble stage (spg_assemble / spg_match_assemble / spg_group_batch; not spg_group_host,
 * which launches per chunk) to publish its own completion: the CTA that finishes last release-stores `value` into
 * *word_dev (local or peer memory) after every record of the launch has been stored -- the producer's "my records
 * have landed" without a separate signalling kernel.  One shot; NULL disarms.  Needs spg_set_wire_output. */
int spg_arm_wire_signal(spg_handle *h, uint64_t *word_dev, uint64_t value);

/* ---- peer memory + stream-ordered signalling for the NVLink gather (no NCCL in the data path) ------------ */
/* A sink is plain device memory that other processes (one per GPU) can map: create it on the owner, send the
 * 64-byte handle to the peers by any means (torch.distributed), open it there.  Zero-filled on creation. */
int spg_wire_create(int32_t device, uint64_t bytes, void **dev_ptr, unsigned char ipc_handle[64]);
int spg_wire_open(int32_t device, const unsigned char ipc_handle[64], void **peer_ptr);
int spg_wire_close(void *peer_ptr);
int spg_wire_destroy(int32_t device, void *dev_ptr);
/* release-store `value` into a 64-bit word (local or peer memory) once everything earlier on `stream` has
 * completed: a one-thread kernel (fence.sys + st.release.sys).  The producer's "my records have landed". */
int spg_wire_signal(int32_t device, uint64_t *word_dev, uint64_t value, void *stream);
/* the same value into up to 32 words (each local or peer memory) with ONE launch: the consumer's acknowledgement to all ranks */
int spg_wire_signal_many(int32_t device, uint64_t *const *words_dev, int32_t n_words, uint64_t value, void *stream);
/* make `stream` wait until *word_dev >= value.  `word_dev` must be LOCAL device memory: the wait is a stream
 * memory operation (cuStreamWaitValue64), executed by the copy/compute front end -- no kernel sits on an SM
 * spinning, so it cannot collide with the persistent kernels that own every SM.  */
int spg_wire_wait(int32_t device, const uint64_t *word_dev, uint64_t value, void *stream);

/* number of kernel launches issued by this handle since creation (bench.py's gpu_launches) */
int64_t spg_launch_count(const spg_handle *h);
/* name of the kernel variant the last launch of a stage used (0 nms_peaks, 1 limb_score, 2 limb_match, 3 assemble,
 * 4 post-network stage);
 * "" before the first launch.  Profiling aid: lets bench.py label its per-kernel numbers with the ncu kernel name. */
const char *spg_stage_kernel(const spg_handle *h, int32_t stage);

#ifdef __cplusplus
}
#endif
#endif /* SPGROUP_H_ */
