/*
 * sva_c_api.h — C ABI of libsva_b200.so: the B200 (sm_100a) implementation of the
 * StereoVisionArray multi-camera depth hot path.
 *
 * Every entry point is `extern "C"`, takes plain pointers + sizes, returns an int status
 * (0 = SVA_OK, negative = sva_status) and never retains a caller pointer after it returns.
 * The reference has no error codes (failures are cv::Exception / UB, SURVEY §8b); the adapter
 * in adapter/sva_functions.cpp turns a non-zero status back into an exception.
 *
 * Citations `file:line` are into the reference tree (Nahuel-M/StereoVisionArray).
 * Images are 8-bit, single channel, row-major: (data, rows, cols, step_bytes) == cv::Mat
 * {data, rows, cols, step}.
 */
#ifndef SVA_C_API_H
#define SVA_C_API_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVA_API_VERSION 1
#define SVA_MAX_PAIRS 32
#define SVA_COST_CAP_MAX 4095      /* PACK_U16 costs live in [0, cap], cap <= 4095 (DESIGN.md §3) */
#define SVA_COST_INVALID_U32 0xFFFFFFFFu
#define SVA_DISP_INVALID 0xFFFFu   /* u16 disparity of a rejected / masked / border pixel */
#define SVA_SUBPIX_INVALID (-1.0f)

typedef enum sva_status {
    SVA_OK = 0,
    SVA_ERR_BAD_ARG = -1,      /* null pointer, non-positive size, unsupported parameter */
    SVA_ERR_ROI = -2,          /* a window leaves the image: the reference would throw cv::Exception (Mat::operator()(Rect)) */
    SVA_ERR_CUDA = -3,         /* CUDA runtime error; text in sva_last_error() */
    SVA_ERR_NO_DEVICE = -4,    /* no sm_100 device: there is NO CPU fallback */
    SVA_ERR_STATE = -5,        /* stage called before the stage that produces its input */
    SVA_ERR_NOMEM = -6,
    SVA_ERR_COMM = -7          /* multi-GPU: NCCL / CUDA-IPC failure, or a neighbour's hand-off did not arrive in time */
} sva_status;

/* enum pairType — include/functions.h:8-19, same values in the same order. */
typedef enum sva_pair_type {
    SVA_ORTHOGONAL = 0, SVA_DIAGONAL = 1, SVA_TO_CENTER = 2, SVA_LINE_HORIZONTAL = 3, SVA_LINE_VERTICAL = 4,
    SVA_CROSS = 5, SVA_JUMP_CROSS = 6, SVA_TO_CENTER_SMALL = 7, SVA_MID_LEFT = 8, SVA_MID_TOP = 9
} sva_pair_type;

/* class Camera — include/Camera.h:6-21: data members in declaration order pos3D, f, pixel_size. */
typedef struct sva_camera {
    double pos[3];
    double f;
    double pixel_size;
} sva_camera;

typedef struct sva_image_u8 {
    const uint8_t* data;
    int32_t rows, cols;
    size_t step; /* bytes between rows */
} sva_image_u8;

/* Parameters of the rectified-array ("volume") formulation; frozen spec in DESIGN.md §3. */
typedef struct sva_params {
    int32_t width, height;
    int32_t num_disp;               /* D; multiple of 8, 8..256 */
    int32_t min_disp;               /* disparity of volume index 0 (delta = min_disp + d) */
    int32_t win_half;               /* k: SAD window is [x-k, x+k) x [y-k, y+k) — src/CameraStereoVision.cpp:44,57,77 */
    int32_t n_pairs;                /* 1..SVA_MAX_PAIRS */
    int32_t pair_gx[SVA_MAX_PAIRS]; /* grid offset of the other camera from the reference camera, in baselines */
    int32_t pair_gy[SVA_MAX_PAIRS]; /* match of ref (x,y) at disparity delta is other (x - gx*delta, y - gy*delta) */
    int32_t cost_shift;             /* PACK_U16: C = min(cost_cap, raw >> cost_shift), applied after the cross-pair sum */
    int32_t cost_cap;               /* 1..SVA_COST_CAP_MAX; also the value of an invalid cell */
    int32_t p1, p2;                 /* SGM penalties, 0 <= p1 <= p2 <= 4095 */
    int32_t n_paths;                /* 0 (no aggregation: WTA on C), 4 or 8 */
    int32_t lr_gx;                  /* 0 = no left-right check; -1/+1 = side of the virtual horizontal other view */
    int32_t lr_max_diff;            /* reject when |d - d_other| > lr_max_diff */
    int32_t subpixel;               /* 0/1: parabolic refinement of the integer winner */
    int32_t reserved[8];            /* reserved[0] = matching cost (sva_cost_mode, default SVA_COST_SAD); the rest must be 0 */
} sva_params;

/* Per-pixel matching cost that K1a sums over the pairs (the box window, shift / cap, SGM and WTA are the same for both).
 * SVA_COST_SAD: |R - I_k| — getAbsDiff, src/functions.cpp:215-218.  SVA_COST_CENSUS: Hamming distance of 9 x 7 census signatures (62 bits;
 * bit = neighbour < centre, out-of-image = 0) — named by north_star, absent from the reference: spec frozen in oracle/sva_oracle.c, parity
 * unpinned by the reference. */
typedef enum sva_cost_mode { SVA_COST_SAD = 0, SVA_COST_CENSUS = 1 } sva_cost_mode;

typedef struct sva_ctx sva_ctx;

/* ---- context ----------------------------------------------------------------------------------------------- */
int sva_create(int device, sva_ctx** out);          /* one ctx per GPU; owns a stream and the HBM workspaces.  SVA_ERR_BAD_ARG when an
                                                        A/B switch (DESIGN §8a) holds a value outside its documented set */
int sva_destroy(sva_ctx* ctx);
const char* sva_last_error(const sva_ctx* ctx);      /* valid until the next call on ctx; NULL: why this thread's last sva_create failed */
int sva_api_version(void);
int sva_set_stream(sva_ctx* ctx, void* cuda_stream); /* run on a caller stream (e.g. torch's; NULL = the legacy default stream); the stream must
                                                       * stay alive until sva_use_own_stream / another sva_set_stream / sva_destroy */
int sva_use_own_stream(sva_ctx* ctx);                 /* back to the ctx's own non-blocking stream */
int sva_get_stream(sva_ctx* ctx, void** out_cuda_stream);  /* the stream the ctx currently runs on (to share it with another ctx) */
int sva_synchronize(sva_ctx* ctx);
int sva_kernel_launches(const sva_ctx* ctx, uint64_t* out_count); /* kernels launched by this ctx so far */
/* Self-check for boxes without compute-sanitizer: device buffers allocated after sva_debug_set_guard(ctx, 1) carry 256 KiB canary bands
 * on both sides and a poisoned (0xCD) payload; sva_debug_check_guards synchronises the device and reports how many buffers are guarded
 * and how many canary bytes were overwritten (any value > 0 is an out-of-bounds write by one of the library's kernels). */
int sva_debug_set_guard(sva_ctx* ctx, int on);
int sva_debug_check_guards(sva_ctx* ctx, int64_t* guarded_buffers, int64_t* bad_bytes);

/* ---- 1:1 shims of the reference's scalar helpers (host side, no GPU work) ------------------------------------ */
/* Camera::project — src/Camera.cpp:15-22 */
int sva_camera_project(const sva_camera* cam, const double pos3d[3], int32_t out_px[2]);
/* Camera::inv_project — src/Camera.cpp:25-33 */
int sva_camera_inv_project(const sva_camera* cam, const int32_t px[2], double out_ray[3]);
/* bresenham — include/functions.h:45, src/functions.cpp:253-321.  Returns the number of points (may exceed cap; only cap are written). */
int sva_bresenham(int32_t ax, int32_t ay, int32_t bx, int32_t by, int32_t* out_xy, int32_t cap);
/* getCameraPairs — include/functions.h:34-36, src/functions.cpp:148-213.  camera_num < 0 = the 2-argument overload. */
int sva_get_camera_pairs(int32_t n_cameras, int32_t pair_type, int32_t camera_num, int32_t* out_pairs, int32_t cap);
/* Generalisation to an arbitrary rows x cols grid (SURVEY §8 a9): pairs {ref, i} for every i != ref (TO_CENTER) or the
 * 8-neighbourhood (TO_CENTER_SMALL), plus the grid offsets (gx, gy) = (col_i - col_ref, row_i - row_ref). */
int sva_grid_pairs(int32_t grid_rows, int32_t grid_cols, int32_t ref_index, int32_t pair_type, int32_t* out_pairs,
                   int32_t* out_gx, int32_t* out_gy, int32_t cap);

/* ---- batched hot path, host buffers in / host buffers out (copies are inside the call) ----------------------- */
/* getAbsDiff — include/functions.h:38, src/functions.cpp:215-218: exact sum |a-b| of two equal-size u8 ROIs. */
int sva_abs_diff_u8(sva_ctx* ctx, const sva_image_u8* a, const sva_image_u8* b, double* out_sum);

/* The reference driver's loop nest — src/CameraStereoVision.cpp:49-95 — as ONE call ("literal mode").
 * images[n_images], cams[n_images]; pairs[2*n_pairs] = {ref, other}; mask may be NULL (= all ones).
 * out_disp: rows x cols u8, zero where the reference leaves the Mat unwritten. */
int sva_match_literal(sva_ctx* ctx, const sva_image_u8* images, const sva_camera* cams, int32_t n_images, const int32_t* pairs,
                      int32_t n_pairs, const sva_image_u8* mask, int32_t win_half, double ray_near, double ray_far, uint8_t* out_disp);

/* shiftPerspectiveWithDisparity — include/functions.h:26, src/functions.cpp:55-77 (gather remap, zero where unwritten). */
int sva_shift_perspective_with_disparity(sva_ctx* ctx, const sva_camera* input_cam, const sva_camera* output_cam,
                                         const sva_image_u8* disparity, const sva_image_u8* image, uint8_t* out);

/* improveWithDisparity — include/functions.h:22, src/functions.cpp:11-52.  cams[2*n] = {cam0, cam1} per other image.
 * Returns SVA_ERR_ROI where the reference would throw (a masked pixel whose 2k x 2k windows leave the image). */
int sva_improve_with_disparity(sva_ctx* ctx, const sva_image_u8* disparity, const sva_image_u8* center, const sva_image_u8* images,
                               const sva_camera* cams, int32_t n, const sva_image_u8* mask, int32_t window_size, uint8_t* out);

/* depth = baseline * f / (disparity * pixel_size) in f64 — src/CameraStereoVision.cpp:47,98-100 (inf where disparity == 0). */
int sva_disparity_to_depth(sva_ctx* ctx, const sva_image_u8* disparity, double baseline, double f, double pixel_size, double* out_depth);

/* ---- consumers of the depth output (SURVEY §8 f2 / f3), f64, bit-exact with the reference's serial loops ---------------------------- */
/* shiftPerspective2 — include/functions.h:24, src/functions.cpp:79-104: forward-warp a depth map into another camera's view; where several
 * sources land on a pixel the one the reference visits last (x outer, y inner) wins; pixels nothing lands on are 0 (uninitialised there). */
int sva_shift_perspective2(sva_ctx* ctx, const sva_camera* input_cam, const sva_camera* output_cam, const double* depth, int32_t rows, int32_t cols,
                           double* out);
/* Points3DToDepthMap — include/functions.h:30, src/functions.cpp:118-133: depth = p.z - camera.z at project(p) + resolution/2; the last
 * point in list order wins; unwritten pixels are 0. */
int sva_points3d_to_depth_map(sva_ctx* ctx, const double* points_xyz, int64_t n_points, const sva_camera* cam, int32_t width, int32_t height, double* out);
/* DepthMapToPoints3D — include/functions.h:32, src/functions.cpp:135-146: one point per pixel with depth > 0.1, in column-major pixel order.
 * *out_count = number of points; at most `cap` are written. */
int sva_depth_map_to_points3d(sva_ctx* ctx, const double* depth, int32_t rows, int32_t cols, const sva_camera* cam, int32_t width, int32_t height,
                              double* out_xyz, int64_t cap, int64_t* out_count);
/* calculateAverageError — include/functions.h:53, src/functions.cpp:348-354: cv::mean(image, mask)[0] of an f64 map (0 for an empty mask).
 * Deterministic summation order; equal to any other order within a few ulp. */
int sva_masked_mean_f64(sva_ctx* ctx, const double* image, int32_t rows, int32_t cols, const sva_image_u8* mask, double* out_mean);
/* getGroups — include/functions.h:28, src/functions.cpp:107-116.  Returns the number of groups. */
int sva_get_groups(int32_t n_cameras, const char* group_type, int32_t* out_pairs, int32_t cap_pairs, int32_t* out_sizes, int32_t cap_groups);

/* ---- ingest (SURVEY §8 f4) ---------------------------------------------------------------------------------------------------------- */
/* resize(img, img, Size(), 0.5, 0.5) — src/CameraStereoVision.cpp:18 (default INTER_LINEAR; for the exact 2x decimation of an even-sized
 * u8 image that is the rounded mean of each 2x2 block).  out: rows/2 x cols/2, tight pitch.  Odd sizes are rejected. */
int sva_resize_half_u8(sva_ctx* ctx, const sva_image_u8* img, uint8_t* out);
/* cv::FileStorage YAML matrices — saveImage / loadImage (key "image") and getIdealRef (key "R"), src/functions.cpp:323-346.
 * dtype 0 = u8, 1 = f64, single channel.  read: out == NULL only queries rows / cols / dtype.  Host side, no GPU work. */
int sva_yaml_write_matrix(const char* path, const char* name, const void* data, int32_t rows, int32_t cols, int32_t dtype);
int sva_yaml_read_matrix(const char* path, const char* name, void* out, int64_t cap_bytes, int32_t* rows, int32_t* cols, int32_t* dtype);

/* The whole volume-mode pipeline (cost volume -> SGM -> WTA/LR/sub-pixel), DESIGN.md §3.
 * others[n_pairs] are the other views in pair order.  out_disp: u16 (min_disp + d, SVA_DISP_INVALID when rejected);
 * out_subpix (may be NULL): f32. */
int sva_depth_from_array(sva_ctx* ctx, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others,
                         const sva_image_u8* mask, uint16_t* out_disp, float* out_subpix);

/* Streaming form for a capture stream (configuration c4: independent frames): submit() returns at once with a ticket; frame t+1's
 * upload overlaps frame t's kernels and frame t-1's download (two frames in flight, double-buffered inputs / outputs inside ctx).
 * Every host buffer of a frame — images and outputs — must stay valid and untouched until sva_stream_wait(ticket) returns; use pinned
 * memory for real overlap.  Results are identical to sva_depth_from_array. */
int sva_stream_submit(sva_ctx* ctx, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                      uint16_t* out_disp, float* out_subpix, int64_t* out_ticket);
int sva_stream_wait(sva_ctx* ctx, int64_t ticket);
/* device-clock stopwatch of the streaming path: elapsed(ticket) = time from the last mark() to the end of that frame's download */
int sva_stream_mark(sva_ctx* ctx);
int sva_stream_elapsed(sva_ctx* ctx, int64_t ticket, float* out_ms);

/* getGroups — include/functions.h:28, src/functions.cpp:107-116: the depth map of every reference view of ONE array frame, in one call.
 * images[n_images]: the frame's cameras on a grid of grid_cols columns (camera i at row i / grid_cols, column i % grid_cols).  The groups come in
 * the layout sva_get_groups writes: pairs[2 * k] = {ref, other} flattened, sizes[g] pairs in group g, every pair of a group with the same
 * reference (the CHESS list goes in unchanged, its duplicate pairs included).  Pair j of group g gets the grid offsets
 * gx = col(other) - col(ref), gy = row(other) - row(ref); p is a template whose n_pairs, pair_gx and pair_gy are zero, every other field
 * applies to every group.  The groups [group_begin, group_end) are computed: out_disp[g - group_begin] (width x height u16) and, when
 * out_subpix and its entry are not NULL, out_subpix[g - group_begin] (f32) receive exactly what sva_depth_from_array returns for that group's
 * parameters, reference view, other views and mask.  masks: NULL, or one per group of the range (data == NULL: no mask).  Only the cameras
 * these groups read need data; the others may have data == NULL, so a rank of a sharded frame passes and uploads only its own cameras.
 * Each camera read is uploaded once; the groups then run through the capture-stream pipeline of sva_stream_submit (frames in flight there
 * complete first, and their tickets stay waitable).  Synchronous: returns once every map is in the caller's buffers.
 * SVA_ERR_BAD_ARG, with nothing enqueued: a group whose pairs do not share one reference, a pair of a camera with itself, an index outside
 * [0, n_images), n_images not a multiple of grid_cols, a group range outside [0, n_groups], a group whose derived parameters are refused
 * (e.g. more than 32 pairs, a window sum that overflows), a camera read by the range without data or not width x height, a mask of the
 * wrong size. */
int sva_depth_groups(sva_ctx* ctx, const sva_params* p, int32_t grid_cols, const sva_image_u8* images, int32_t n_images, const int32_t* pairs,
                     const int32_t* sizes, int32_t n_groups, int32_t group_begin, int32_t group_end, const sva_image_u8* masks,
                     uint16_t* const* out_disp, float* const* out_subpix);

/* ---- multi-view depth fusion (DESIGN.md §3 item 6): the maps of several reference views of one array frame merged into one camera's view ----
 * No reference counterpart (shiftPerspective2 warps f64 metric depth with "last writer wins"); spec frozen in tests/fuse_oracle.c
 * (orc_fuse_views), parity unpinned by the reference.  Everything after the fixed-point step is integer: the result is bit-exact and does not
 * depend on the order of the views.
 *  1. pixel (x, y) of view g is used iff disp != SVA_DISP_INVALID and, with sub-pixel maps, 0 <= subpix < 4352; q = 16 * disp, or with
 *     sub-pixel maps q = rint(16 * subpix) (ties to even), in 1/16 px;
 *  2. it lands on x' = x - ((gx * q + 8) >> 4), y' = y - ((gy * q + 8) >> 4) of the target, (gx, gy) = (col t - col r_g, row t - row r_g),
 *     >> an arithmetic (floor) shift; outside the image it is dropped;
 *  3. per view and target pixel the largest q that lands there wins (the nearest surface);
 *  4. among the views' candidates c_h at a pixel, c* has the largest support #{h : |c_h - c*| <= tol_16} (ties: the larger value);
 *     M = {h : |c_h - c*| <= tol_16}, n* = |M|, q^ = (sum_M c_h + n* / 2) / n*;
 *  5. rejected (no candidate, n* < min_support, or target mask 0): disp = SVA_DISP_INVALID, subpix = -1; accepted: disp = (q^ + 8) >> 4,
 *     subpix = q^ / 16.  support = n* everywhere (0 without a candidate). */
typedef struct sva_fuse_params {
    int32_t tol_16;       /* candidates within tol_16 / 16 px agree; 0..4095 */
    int32_t min_support;  /* views that must agree for a pixel to be accepted; 1..n_views */
    int32_t reserved[6];  /* must be 0 */
} sva_fuse_params;
/* The maps in host memory (e.g. sva_depth_groups' outputs, or maps gathered from the ranks of a sharded frame): disp[g] (and subpix[g] when
 * subpix is not NULL) width x height of the view whose reference camera is view_refs[g], on a grid of grid_cols columns; target: the camera
 * whose view the result is in; target_mask: NULL or width x height (0 = reject).  out_subpix and out_support (u8) may be NULL.  Synchronous.
 * SVA_ERR_BAD_ARG, with nothing enqueued: n_views outside 1..32, a reference or the target outside [0, n_cameras), n_cameras not a positive
 * multiple of grid_cols, tol_16 outside 0..4095, min_support outside 1..n_views, non-zero reserved fields, a null map or output, a size below
 * 1 x 1, a mask of the wrong size. */
int sva_fuse_maps(sva_ctx* ctx, int32_t width, int32_t height, int32_t grid_cols, int32_t n_cameras, const int32_t* view_refs, int32_t n_views,
                  const uint16_t* const* disp, const float* const* subpix, int32_t target, const sva_fuse_params* f,
                  const sva_image_u8* target_mask, uint16_t* out_disp, float* out_subpix, uint8_t* out_support);
/* Every group of the frame (sva_depth_groups over [0, n_groups)), then their fusion into camera target, in one call: each group's maps are
 * warped into the target's view on the device right after its K3 and never leave it; the fused maps are the only download.  The views are the
 * groups (view_refs = each group's reference camera, n_cameras = n_images); the sub-pixel maps are used iff p->subpixel == 1.  The result
 * equals sva_depth_groups followed by sva_fuse_maps on its outputs bit for bit.  SVA_ERR_BAD_ARG, with nothing enqueued: every refusal of
 * both calls. */
int sva_depth_groups_fused(sva_ctx* ctx, const sva_params* p, int32_t grid_cols, const sva_image_u8* images, int32_t n_images,
                           const int32_t* pairs, const int32_t* sizes, int32_t n_groups, const sva_image_u8* masks, int32_t target,
                           const sva_fuse_params* f, const sva_image_u8* target_mask, uint16_t* out_disp, float* out_subpix,
                           uint8_t* out_support);

/* ---- staged, device-resident form of the same pipeline (what bench.py times with inputs already in HBM) ------- */
typedef enum sva_stage {
    SVA_STAGE_AD = 1,        /* K1a: A(y,x,d) = sum_k |R - I_k(shifted)|            -> u16 [H][W][D] */
    SVA_STAGE_BOX = 2,       /* K1b: 2k x 2k box sum + shift/cap + validity          -> u16 [H][W][D] (C) */
    SVA_STAGE_SGM = 3,       /* K2 then K3 (WTA / LR / sub-pixel): S and the outputs -> u16 [H][W][D], disparity maps */
    SVA_STAGE_ALL = 100
} sva_stage;

int sva_frame_upload(sva_ctx* ctx, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask);
/* pair subset [pair_begin, pair_end) for SVA_STAGE_AD (pair sharding, SURVEY §8e); pass 0, n_pairs for everything. */
int sva_frame_set_pair_range(sva_ctx* ctx, int32_t pair_begin, int32_t pair_end);
int sva_frame_run(sva_ctx* ctx, int32_t stage);
/* CUDA-event time of `iters` back-to-back runs of `stage` on the ctx stream, in milliseconds (total, not mean). */
int sva_frame_time(sva_ctx* ctx, int32_t stage, int32_t iters, float* out_ms);
/* Runs `stage` once with a CUDA-event pair around every kernel: names[i] (static strings) / ms[i]; returns the kernel count. */
int sva_frame_kernel_times(sva_ctx* ctx, int32_t stage, const char** names, float* ms, int32_t cap);
/* sva_frame_time with an event pair around every kernel: per distinct kernel name, the summed time and the launch count. */
int sva_frame_time_detailed(sva_ctx* ctx, int32_t stage, int32_t iters, float* out_total_ms, const char** names, float* sum_ms,
                            int32_t* counts, int32_t cap);
/* CUDA-event stopwatch on the ctx stream: times a sequence of host-buffer calls (the end-to-end path) on the device clock. */
int sva_timer_start(sva_ctx* ctx);
int sva_timer_stop(sva_ctx* ctx, float* out_ms);
/* Test hooks: store_full_s != 0 makes the last SGM pass also write S_total; sgm_dir_mask != 0 runs exactly those path
 * directions (bit i = direction i of {v+, v-, h+, h-, d++, d-+, d+-, d--}) as accumulate passes and skips the final pass. */
int sva_frame_set_debug(sva_ctx* ctx, int32_t store_full_s, uint32_t sgm_dir_mask);
/* After an external (cross-GPU) reduction has written the complete A volume into sva_frame_ad_device_ptr()'s buffer. */
int sva_frame_mark_ad_ready(sva_ctx* ctx);
int sva_frame_download_ad(sva_ctx* ctx, uint16_t* out);         /* [H][W][D] */
int sva_frame_download_cost(sva_ctx* ctx, uint16_t* out);       /* [H][W][D] */
int sva_frame_download_raw_cost(sva_ctx* ctx, uint32_t* out);   /* RAW_U32 recomputed from A: [H][W][D] */
int sva_frame_download_sgm(sva_ctx* ctx, uint16_t* out);        /* S [H][W][D]: the sum of all n_paths paths (or of the debug direction mask) */
int sva_frame_download_disparity(sva_ctx* ctx, uint16_t* out_disp, float* out_subpix);
/* Device pointer + byte size of the A volume, so a caller can reduce it across GPUs (NCCL via torch.distributed). */
int sva_frame_ad_device_ptr(sva_ctx* ctx, void** out_ptr, size_t* out_bytes);

/* ---- multi-GPU building blocks for ONE frame sharded by disparity slices, path directions and row blocks (DESIGN.md §7) ----------
 * Rank r of G uploads the frame with num_disp = D/G and min_disp = dmin + r*D/G and runs SVA_STAGE_AD + SVA_STAGE_BOX: that is its slice of
 * the cost volume, complete, with no cross-GPU reduction.  The caller all-gathers the slices into a slice-major device volume
 * [G][H][W][D/G], switches every rank to the full range with sva_frame_set_params, lets each rank aggregate its share of the path directions
 * (sva_frame_sgm_directions: the result is that rank's partial S over `rows_alloc` >= H rows, rows beyond H zero), reduce-scatters the
 * partial sums by row blocks and runs K3 per block (sva_frame_wta_rows; the left-right check is row-local). */
int sva_frame_cost_device_ptr(sva_ctx* ctx, void** out_ptr, size_t* out_bytes);  /* C [H][W][D] of the current parameters */
/* Same images and mask, new parameters.  The views were staged at upload for that upload's pairs and disparity reach: SVA_STAGE_AD runs
 * again only if pairs, min_disp and win_half are unchanged and num_disp does not reach further (else SVA_ERR_STATE: upload again); any
 * parameter set may be used for the stages after K1a (the full range after a disparity-slice cost volume). */
int sva_frame_set_params(sva_ctx* ctx, const sva_params* p);
/* dir_mask bit i = direction i of {v+, v-, h+, h-, d++, d-+, d+-, d--}; slice_disp = D/G for a slice-major volume, 0 for [H][W][D] */
int sva_frame_sgm_directions(sva_ctx* ctx, const void* cost_dev, int32_t slice_disp, uint32_t dir_mask, int32_t rows_alloc, void** out_s_ptr,
                             size_t* out_bytes);
int sva_frame_wta_rows(sva_ctx* ctx, const void* s_rows_dev, int32_t y0, int32_t rows);  /* s_rows_dev = image rows [y0, y0+rows) of S (NULL: the ctx's own S) */
int sva_frame_download_disparity_rows(sva_ctx* ctx, int32_t rows, uint16_t* out_disp, float* out_subpix);

/* ---- building blocks for ONE frame sharded by ROW BLOCKS end to end (DESIGN.md §7): no volume ever crosses GPUs -------------------------
 * Rank r owns image rows [y0, y0 + rows).  sva_frame_rows_begin zeroes those rows of the aggregation volume.  sva_frame_sgm_rows runs one
 * direction group on the block: group 2 = {h+, h-} (local), group 0 = {v+, d++, d-+} sweeping down, group 1 = {v-, d+-, d--} sweeping up.
 * A row-sweeping group continues the path lines of the block above (below): state_in / state_out are device buffers of 3 * W * D u16
 * holding L of every line after the neighbouring block's last row / after this block's last row (NULL at the sweep's first / last block);
 * the caller moves them between GPUs (a few MB per hop).  sva_frame_wta_rows(ctx, NULL, y0, rows) then runs K3 on the block. */
int sva_frame_rows_begin(sva_ctx* ctx, int32_t y0, int32_t rows);
int sva_frame_sgm_rows(sva_ctx* ctx, int32_t group, int32_t y0, int32_t rows, const void* state_in, void* state_out);

/* ---- multi-GPU from C (SURVEY §8b / §8e): one process per GPU, one context per process and GPU ------------------------------------------
 * The reference has no counterpart (it is single-threaded, SURVEY §0.1); the sharding units are its own loops: the PAIR loop
 * src/CameraStereoVision.cpp:55 over the pair list of getCameraPairs (include/functions.h:34-36, src/functions.cpp:150-155), and the
 * pixel-ROW loop src/CameraStereoVision.cpp:49.
 *
 * Communicator: NCCL, loaded at run time with dlopen("libnccl.so.2") (the library has no link-time dependency on it).  Rank 0 calls
 * sva_comm_get_unique_id and hands the 128 bytes to the other ranks by any means (MPI, a file, torch.distributed ...); every rank then
 * calls sva_comm_init (collective). */
#define SVA_COMM_ID_BYTES 128
#define SVA_IPC_HANDLE_BYTES 64
int sva_comm_get_unique_id(uint8_t out_id[SVA_COMM_ID_BYTES]);
int sva_comm_init(sva_ctx* ctx, const uint8_t id[SVA_COMM_ID_BYTES], int32_t rank, int32_t world);
int sva_comm_destroy(sva_ctx* ctx);
int sva_comm_barrier(sva_ctx* ctx);  /* all ranks' ctx streams meet (one-word all-reduce), then the host waits for its stream */
/* Pair sharding, the scheme north_star names: after SVA_STAGE_AD over this rank's pair range (sva_frame_set_pair_range) the partial AD
 * volumes are sum-reduced onto `root` as packed u32 — NCCL has no 16-bit integer type, and a cell's total is <= 255 * 32 < 2^16, so no carry
 * crosses the half-word: bit-exact in any order.  On root the volume is then complete (as after SVA_STAGE_AD over all pairs). */
int sva_frame_reduce_ad(sva_ctx* ctx, int32_t root);
/* The whole pair-sharded frame in one collective call: upload everywhere, K1a over the rank's pairs (balanced contiguous ranges, e.g. 15
 * pairs over 8 ranks = 2,2,2,2,2,2,2,1), reduce, and on root K1b + SGM + K3 and the download (out_* are ignored elsewhere). */
int sva_depth_pair_sharded(sva_ctx* ctx, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                           int32_t root, uint16_t* out_disp, float* out_subpix);

/* Row-block pipeline with PEER-DIRECT hand-off (DESIGN.md §7): rank r owns image rows [r * ceil(H / G), ...), computes their cost volume and
 * horizontal paths locally, and continues the row-sweeping path lines of its neighbour: the march kernel of the block above (below) stores L
 * of every line after its last row STRAIGHT INTO THIS rank's state buffer over NVLink (a peer-mapped pointer), a flag kernel publishes the
 * frame's sequence number, and a wait kernel on this rank's stream holds the next march until it is there — no host in the loop, no NCCL on
 * the data path.  sva_rows_run only enqueues; several contexts per GPU (each with its own link) keep several frames in flight.
 *   sva_rows_open      allocates the link memory (two state buffers of 3 * W * D u16 and the flags) for this geometry and rank
 *   sva_rows_export / sva_rows_connect    CUDA-IPC handle of the link memory out / the neighbours' handles in (NULL at the array's ends)
 *   sva_rows_connect_comm                 the same exchange over the context's communicator (collective)
 *   sva_rows_connect_local                neighbours that live in the same process (tests; one process driving several GPUs)
 *   sva_rows_run       enqueue this rank's part of the uploaded frame (K1a, K1b, horizontal paths, both sweeps, K3 on the block)
 *   sva_rows_download  wait for it; SVA_ERR_COMM if a hand-off did not arrive within SVA_ROWS_TIMEOUT_MS (default 20000) */
int sva_rows_open(sva_ctx* ctx, const sva_params* p, int32_t rank, int32_t world);
int sva_rows_export(sva_ctx* ctx, uint8_t out_handle[SVA_IPC_HANDLE_BYTES]);
int sva_rows_connect(sva_ctx* ctx, const uint8_t* prev_handle, const uint8_t* next_handle);
int sva_rows_connect_comm(sva_ctx* ctx);
int sva_rows_connect_local(sva_ctx* ctx, sva_ctx* prev, sva_ctx* next);
int sva_rows_block(const sva_ctx* ctx, int32_t* out_y0, int32_t* out_rows);
int sva_rows_run(sva_ctx* ctx);
/* The same frame in two parts (phase 0: cost volume, horizontal paths, the sweep that reaches this rank first; phase 1: the other sweep and
 * K3), for hosts that keep several frames in flight: several contexts share ONE stream (sva_get_stream / sva_set_stream) and the host
 * enqueues phase 0 of frame f, then phase 1 of frame f - P + 1 — frames overlap across GPUs without two big kernels ever running at once. */
int sva_rows_run_phase(sva_ctx* ctx, int32_t phase);
/* The same frame in three parts, for hosts with three or more frames in flight: part 0 = cost volume (+ horizontal paths on the ranks that do
 * not start a sweep) — nothing in it waits for a neighbour; part 1 = the first sweep (+ horizontal paths on the two ranks that start one);
 * part 2 = the other sweep and K3.  Enqueued as part 0 of frame f, part 1 of frame f - 1, part 2 of frame f - P + 1, every wait for a
 * neighbour's state sits behind work of a later frame that needs no neighbour.  (sva_rows_run_phase: phase 0 = parts 0 + 1, phase 1 = part 2.) */
int sva_rows_run_part(sva_ctx* ctx, int32_t part);
int sva_rows_download(sva_ctx* ctx, uint16_t* out_disp_rows, float* out_subpix_rows);  /* the block's rows; out_subpix_rows may be NULL */
int sva_rows_close(sva_ctx* ctx);
/* one synchronous call per frame: upload + sva_rows_run + sva_rows_download */
int sva_depth_rows_sharded(sva_ctx* ctx, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                           uint16_t* out_disp_rows, float* out_subpix_rows);

/* ---- a STREAM of frames through the row-block pipeline, one call per frame and rank (DESIGN.md §7) --------------------------------------
 * The order skewed by chain position behind one call.  The stream borrows world + 1 contexts of this rank: each has been through
 * sva_rows_open(p, rank, world) with the same rank, world and geometry, all run on ONE stream (sva_get_stream), and context j of every rank forms
 * one chain.  Their links are connected before the first submit: with sva_rows_connect / sva_rows_connect_local before or after create, or with
 * sva_rows_stream_connect_comm (collective: one all-gather of all world + 1 handles per rank over ctxs[0]'s communicator; nothing to do for a
 * world of one).  Errors are reported through sva_last_error(ctxs[0]); a refused call enqueues nothing.  The stream does not own the contexts:
 * flush, wait and destroy it before them.
 *
 * Submit number i (its ticket) is iteration i of the skewed order: part 0 of frame i, part 1 of frame i - 1 - min(r, G-1-r) and part 2 of frame
 * i - 1 - max(r, G-1-r) (sva_rows_run_part), frame f on context f mod (world + 1).  flush enqueues the remaining iterations, after which every
 * submitted frame completes; a submit after a flush starts a new fill, tickets continuing.  Every rank makes the same sequence of submit and
 * flush calls.
 *
 * The images are uploaded on a copy stream of the object once the cost volume of the context's previous frame has read its own, the mask once
 * that frame's K3 has; the block's rows come back on a second copy stream, through pinned staging owned by the object: a ring of world + 2
 * slots, one per ticket.  The maps reach out_disp_rows / out_subpix_rows (rows x width of sva_rows_block;
 * out_subpix_rows may be NULL) in sva_rows_stream_wait(ticket) or when the ticket's slot is reused, whichever comes first: the ticket is then
 * retired, and until then the caller's input images and output buffers must stay valid and untouched.
 * With pinned inputs, submit never waits for device work of the current or the previous iteration: it waits only when it reuses a slot, for
 * the download of a frame at least two iterations old.  With pageable inputs cudaMemcpy2DAsync may hold the host until the context's previous
 * frame has finished — safe in the skewed order, but the upload then no longer overlaps the iteration: pin the images for real overlap.
 * Nothing is allocated on the device after create (which warms every context up for the geometry, masked and unmasked).
 *
 * sva_rows_stream_wait: SVA_ERR_STATE while the ticket's last part is not enqueued yet (submit more frames, or flush); SVA_ERR_COMM if a
 * hand-off of the frame's context timed out (SVA_ROWS_TIMEOUT_MS) up to that frame — the maps are then not valid; SVA_ERR_BAD_ARG for a ticket
 * never issued.  A retired ticket returns at once. */
typedef struct sva_rows_stream sva_rows_stream;
int sva_rows_stream_create(sva_ctx* const* ctxs, int32_t n_ctxs, const sva_params* p, sva_rows_stream** out);
int sva_rows_stream_connect_comm(sva_rows_stream* s);
int sva_rows_stream_submit(sva_rows_stream* s, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                           uint16_t* out_disp_rows, float* out_subpix_rows, int64_t* out_ticket);
int sva_rows_stream_flush(sva_rows_stream* s);
int sva_rows_stream_wait(sva_rows_stream* s, int64_t ticket);
int sva_rows_stream_destroy(sva_rows_stream* s);  /* waits for the work in flight; tickets not yet retired are dropped */

#ifdef __cplusplus
}
#endif
#endif /* SVA_C_API_H */
