/* dfsfm_b200 -- C ABI of the B200-native dense-matching engine for DetectorFreeSfM's two hot paths.
 *
 * Plain pointers and sizes only; every pointer named *_dev is a CUDA device pointer on the engine's device, every
 * `stream` is a cudaStream_t passed as void*.  All functions return 0 on success and a non-zero code on failure;
 * dfsfm_last_error() then returns a description (thread-local).  No exception crosses this boundary, nothing here
 * falls back to the CPU.
 *
 * Reference interfaces replaced (paths relative to zju3dv/DetectorFreeSfM):
 *   HP-1  third_party/LoFTR/src/loftr/loftr.py:29-81  LoFTR.forward, called from
 *         src/coarse_match/coarse_match_worker.py:94-100 (extract_matches) behind the NEUSFM_coarse_matcher hook.
 *   HP-2  src/MultiviewMatcher/MultiviewMatcher.py:59-405  MultiviewMatcher.forward, called from
 *         src/post_optimization/matcher_model/multiview_match_worker.py:59-64 (extract_results) per refinement chunk.
 *   L0    third_party/RoIAlign.pytorch/roi_align/src/crop_and_resize_gpu.cpp:18-61 crop_and_resize_gpu_forward.
 */
#ifndef DFSFM_B200_H_
#define DFSFM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* dfsfm_last_error(void);
int dfsfm_version(void);

/* ------------------------------------------------------------------------------------------------ HP-1: coarse matcher */
typedef struct dfsfm_coarse dfsfm_coarse_t;

/* LoFTR(config) construction (loftr.py:12-27).  d_model=256, nhead=8, 8 layers ['self','cross']*4 (default.py:14-24). */
int dfsfm_coarse_create(dfsfm_coarse_t** out, int device);
void dfsfm_coarse_destroy(dfsfm_coarse_t* h);

/* Upload one packed parameter (host fp32, row-major [rows][cols]).  kind 0: matrix stored as split-fp16 GEMM operand,
 * kind 1: fp32 vector/table.  Names and packing: detectorfreesfm_b200/packing.py (state_dict -> BN-folded operands). */
int dfsfm_coarse_set_param(dfsfm_coarse_t* h, const char* name, const float* host, int64_t rows, int64_t cols, int kind);

/* ResNetFPN_8_2 (coarse sub-graph) + PositionEncodingSine + 'n c h w -> n (h w) c'  (loftr.py:45-59):
 * image_dev [H][W] fp32 in [0,1] (H, W multiples of 8), pe_dev [(H/8)*(W/8)][256] fp32,
 * tokens_out_dev [(H/8)*(W/8)][256] fp32.  Exact per image, hence cacheable across pairs. */
int dfsfm_coarse_features(dfsfm_coarse_t* h, const float* image_dev, int H, int W, const float* pe_dev, float* tokens_out_dev,
                          void* stream);

/* Same for the two images of a pair (both H x W) in one launch per layer -- the backbone kernels get twice the tiles to spread
 * over the SMs.  tokens*_out_dev [(H/8)*(W/8)][256] fp32, bitwise equal to two dfsfm_coarse_features calls. */
int dfsfm_coarse_features_pair(dfsfm_coarse_t* h, const float* image0_dev, const float* image1_dev, int H, int W, const float* pe_dev,
                               float* tokens0_out_dev, float* tokens1_out_dev, void* stream);

/* Same, plus the FPN top-down path to the 1/2-resolution fine map x1_out (resnet_fpn.py:110-118, match type 'coarse_fine'):
 * feat_f_out_dev [(H/2)*(W/2)][128] fp32 (NHWC rows). */
int dfsfm_coarse_features_fine(dfsfm_coarse_t* h, const float* image_dev, int H, int W, const float* pe_dev, float* tokens_out_dev,
                               float* feat_f_out_dev, void* stream);

/* FinePreprocess.forward + loftr_fine + FineMatching.forward (loftr_module/fine_preprocess.py:29-59, transformer.py:80-101 with
 * d_model 128 / 2 layers, utils/fine_matching.py:15-61) for the M coarse matches (i_ids, j_ids):
 * feat_f*: fine maps [Hf*Wf][128]; feat_c*: coarse tokens AFTER the coarse transformer; w*c: coarse grid widths.
 * coords_out_dev [M][2] = coords_normed * (W // 2) (multiply by scale * scale1 to get the mkpts1_f offset, fine_matching.py:70-72);
 * std_out_dev [M] (expec_f[:, 2]). */
int dfsfm_coarse_fine_match(dfsfm_coarse_t* h, const float* feat_f0_dev, int Hf0, int Wf0, const float* feat_f1_dev, int Hf1, int Wf1,
                            const float* feat_c0_dev, int w0c, const float* feat_c1_dev, int w1c, const int32_t* i_ids_dev,
                            const int32_t* j_ids_dev, int M, float* coords_out_dev, float* std_out_dev, void* stream);

/* LocalFeatureTransformer.forward (loftr_module/transformer.py:80-101), in place on feat0_dev [L][256], feat1_dev [S][256]. */
int dfsfm_coarse_transformer(dfsfm_coarse_t* h, float* feat0_dev, int L, float* feat1_dev, int S, void* stream);

/* CoarseMatching.forward + get_coarse_match (utils/coarse_matching.py:84-258, dual-softmax, inference, no padding masks):
 * writes up to `capacity` matches in ascending i order: i_ids/j_ids int32, mconf fp32, and their number to n_matches_dev.
 * conf_out_dev: optional dense [L][S] confidence matrix (NULL in production). */
int dfsfm_coarse_match(dfsfm_coarse_t* h, const float* feat0_dev, int h0c, int w0c, const float* feat1_dev, int h1c, int w1c, float thr,
                       int border_rm, float temperature, int32_t* i_ids_dev, int32_t* j_ids_dev, float* mconf_dev,
                       int32_t* n_matches_dev, int capacity, float* conf_out_dev, void* stream);

/* ---------------------------------------------------------------------------------- L0: RoIAlign (crop_and_resize) */
/* crop_and_resize_gpu_forward (crop_and_resize_gpu.cpp:18-61): image NCHW fp32, boxes [n][4] = (y1,x1,y2,x2) normalised,
 * box_index [n] int32, crops [n][C][crop_h][crop_w] fp32. */
int dfsfm_crop_and_resize_forward(const float* image_dev, int batch, int depth, int image_h, int image_w, const float* boxes_dev,
                                  const int32_t* box_index_dev, int num_boxes, float extrapolation_value, int crop_h, int crop_w,
                                  float* crops_dev, void* stream);

/* ------------------------------------------------------------------------------------------ HP-2: refinement matcher */
typedef struct dfsfm_refine dfsfm_refine_t;

/* MultiviewMatcher(config, test=True) (MultiviewMatcher.py:17-57) with window W, left window LW
 * (multiview_match_worker.py:20-34 rescales them per refinement iteration). */
int dfsfm_refine_create(dfsfm_refine_t** out, int device, int window, int left_window);
void dfsfm_refine_destroy(dfsfm_refine_t* h);
int dfsfm_refine_set_param(dfsfm_refine_t* h, const char* name, const float* host, int64_t rows, int64_t cols, int kind);

/* MultiviewMatcher.forward on one chunk (MultiviewMatcher.py:59-405, n_steps=1, chunk_backbone_img path).
 * images_dev[i]: [3][H_i][W_i] fp32 RGB;  scales_hw [n_img][2] host (h, w ratios);  M tracks, Nq = n_view-1 query slots.
 * query_pts [M][2], ref_pts [Nq][M][2], valid [Nq][M] (uint8), q_img_idx [M], r_img_idx [Nq][M] (-1 = pad), movable [M]:
 * all HOST arrays (the per-chunk dict of construct_matching_data.py:317-476).
 * Outputs (HOST): query_refined [M][2], ref_refined [Nq][M][2], std_out [Nq][M]. */
int dfsfm_refine_chunk(dfsfm_refine_t* h, int n_img, const float* const* images_dev, const int32_t* H, const int32_t* W,
                       const float* scales_hw, int M, int Nq, const float* query_pts, const float* ref_pts, const uint8_t* valid,
                       const int32_t* q_img_idx, const int32_t* r_img_idx, const uint8_t* movable, float* query_refined,
                       float* ref_refined, float* std_out, void* stream);

/* ---------------------------------------------------------------------- match -> keypoint -> index post-processing
 * Replaces the per-image Python of src/coarse_match/coarse_match.py:203-237 (Match2Kpts, keypoint_worker with
 * agg_groupby_2d = np.unique + np.bincount + sorted, update_matches, transform_keypoints;
 * src/coarse_match/coarse_match_worker.py:151-270, src/coarse_match/utils/merge_kpts.py:4-44).
 *   rows_dev        [n_rows][5] fp32: x0, y0, x1, y1, conf of every match, pairs concatenated in matches-dict order
 *   pair_offset_dev [n_pairs+1] first row of every pair (last entry = n_rows)
 *   pair_images_dev [n_pairs][2] index (into the image list) of the pair's first / second image
 * Outputs (device; capacity 2*n_rows key points):
 *   kpt_xy_dev [K][2] fp32 truncated coordinates, kpt_score_dev [K] fp32 summed confidence, images concatenated in list
 *   order, inside an image ordered by descending fp64 score then (x, y) -- the reference's keypoint ids;
 *   image_offset_dev [n_images+1] first key point of every image; match_ids_dev [n_rows][2] int32 keypoint ids (local to
 *   the image) of the two end points of every match.  *n_keypoints = K.  Synchronises the stream. */
typedef struct dfsfm_post dfsfm_post_t;
int dfsfm_post_create(dfsfm_post_t** out, int device);
void dfsfm_post_destroy(dfsfm_post_t* h);
int dfsfm_post_merge_keypoints(dfsfm_post_t* h, const float* rows_dev, int64_t n_rows, int n_pairs, const int64_t* pair_offset_dev,
                               const int32_t* pair_images_dev, int n_images, float* kpt_xy_dev, float* kpt_score_dev,
                               int32_t* image_offset_dev, int32_t* match_ids_dev, int64_t* n_keypoints, void* stream);

/* ---------------------------------------------------------------------- host image pipeline, device part
 * The PIL-LANCZOS resize + /255 of read_grayscale (src/dataset/utils.py:137-148, resize_image :161-177 with interp
 * "pil_LANCZOS"; grayscale2tensor :56-57).  img_dev: uint8 [h][ld] grayscale (cv2.IMREAD_GRAYSCALE).  The fixed-point tables
 * are Pillow's (Resample.c precompute_coeffs + normalize_coeffs_8bpc; built on the host by image_pipeline.lanczos_coeffs):
 * bounds [out][2] = (first input index, tap count), coef [out][ksize] int32 with 22 fractional bits; pass null tables for a
 * dimension that keeps its size (Pillow skips that pass).  tmp_dev: h*out_w bytes when both passes run.
 * out_dev: fp32 [out_h][out_w] = resized uint8 / 255 -- bit-identical to the reference's tensor. */
int dfsfm_resize_lanczos_gray(const uint8_t* img_dev, int h, int w, int64_t ld, const int32_t* xbounds_dev, const int32_t* xcoef_dev, int xksize,
                              const int32_t* ybounds_dev, const int32_t* ycoef_dev, int yksize, int out_h, int out_w, uint8_t* tmp_dev,
                              float* out_dev, void* stream);

/* --------------------------------------------------------------------- SURVEY 8(f) row 2: bag assignment + chunking (host) */
/* FeatureTrackStatus / assign_bags / chunk_bags of src/post_optimization/data_construct/construct_matching_data.py:10-261 and
 * chunks_balance (src/utils/ray_utils.py:100-108) on flat arrays; all pointers are HOST pointers.
 *   tracks   n_tracks feature tracks in the order of point_cloud_assigned_imgID_kptID: track_ids (point3D ids), ref_img_ids (assigned
 *            reference image), obs_offset [n_tracks+1] / obs_img_ids: the raw point3D.image_ids of every track (duplicates included);
 *   frames   keyframe_dict as CSR: frame_img_ids [n_frames], frame_offset [n_frames+1], frame_track_ids (point3D ids whose reference
 *            node lies on the image, key-point order);
 *   max_track_length, max_num_img_in_bag (<= 0: = max_track_length), chunk (tracks per chunk; <= 0: no chunking).
 * The result handle holds the CHUNKED bags in the reference's order (incl. CPython's set iteration order of the image ids). */
typedef struct dfsfm_bags dfsfm_bags_t;
int dfsfm_assign_bags(dfsfm_bags_t** out, int64_t n_tracks, const int64_t* track_ids, const int64_t* ref_img_ids, const int64_t* obs_offset,
                      const int64_t* obs_img_ids, int64_t n_frames, const int64_t* frame_img_ids, const int64_t* frame_offset,
                      const int64_t* frame_track_ids, int max_track_length, int max_num_img_in_bag, int chunk);
void dfsfm_bags_sizes(const dfsfm_bags_t* h, int64_t* n_bags, int64_t* n_bag_images, int64_t* n_tracks, int64_t* n_query);
/* bag_img_off [n_bags+1] / bag_img; bag_trk_off [n_bags+1] / trk_id, trk_ref [n_tracks]; trk_q_off [n_tracks+1] / trk_q */
void dfsfm_bags_export(const dfsfm_bags_t* h, int64_t* bag_img_off, int64_t* bag_img, int64_t* bag_trk_off, int64_t* trk_id, int64_t* trk_ref,
                       int64_t* trk_q_off, int64_t* trk_q);
void dfsfm_bags_destroy(dfsfm_bags_t* h);
/* test hook: one CPython-set expression on small integers, result in iteration order (see csrc/bag_assign.cpp) */
int dfsfm_debug_pyset(int op, const int64_t* a, int64_t na, const int64_t* b, int64_t nb, int64_t* out, int64_t* n_out);

/* -------------------------------------------------------------------------------------------------- test / bench hooks */
/* Shifted-row GEMM engine on raw split-fp16 operands: out[M][N] fp32 = sum_t A[p+shift_t, :cpad] . W[n, t*cpad : (t+1)*cpad].
 * a_dev: [2][a_rows][C] halves, w_dev: [2][w_rows][taps*cpad] halves.  bn in {64,128,208,256}; split in {0,1}. */
int dfsfm_debug_gemm(const void* a_dev, int64_t a_rows, int C, const void* w_dev, int64_t w_rows, int taps, const int32_t* shifts,
                     int cpad, int bn, int split, float* out_dev, int M, int N, void* stream);
/* Same for the tap-group variant (groups of 3 taps with consecutive row shifts share one activation slab); bn in {64,128}. */
int dfsfm_debug_gemm_slab(const void* a_dev, int64_t a_rows, int C, const void* w_dev, int64_t w_rows, int taps, const int32_t* shifts,
                          int cpad, int bn, int bo_mode, float* out_dev, int M, int N, void* stream);
/* GEMM engine variant: 2 = persistent CTA pairs (cta_group::2, default), 1 = one CTA per output tile.  Test hook. */
void dfsfm_set_engine(int version);
int dfsfm_get_engine(void);
/* Per-launch CUDA-event timing for bench.py's roofline attribution: enable(1) clears and starts collecting, enable(0) stops;
 * report() synchronises the device and writes "label count total_ms" lines. Never on inside a timed region. */
void dfsfm_profile_enable(int on);
int dfsfm_profile_report(char* buf, int cap);
/* In-kernel timeline of the engine-2 GEMM (tuning aid): arm(n) makes each of the next n launches record 16 %globaltimer stamps
 * per CTA (0 entry, 1 set-up done, 2 dependency wait over, 3 first operands landed, 4/5 MMAs of first/last tile issued,
 * 6/8 accumulator of first/last tile complete, 7/9 its epilogue done, 10 all roles done, 11 exit); read() synchronises and
 * copies stamps[launch][148][16] and info[launch][2] = {CTAs, tiles}; returns the number of launches captured. */
int dfsfm_debug_timeline_arm(int max_launches);
int dfsfm_debug_timeline_read(uint64_t* stamps, int32_t* info, int max_launches);
/* Number of kernels launched by this library since load (bench.py reports it as gpu_launches). */
int64_t dfsfm_launch_count(void);
/* Programmatic dependent launch for the launches made from the CALLING host thread: 1 on, 0 off, -1 the process default (on; DFSFM_PDL=0
 * turns it off).  A pair worker of a several-workers-per-GPU pool (coarse_match.py:49-55, n_gpus_per_worker 0.5) turns it off: early-resident
 * dependent CTAs would hold SMs another worker's kernel could use. */
void dfsfm_thread_set_pdl(int mode);

#ifdef __cplusplus
}
#endif
#endif /* DFSFM_B200_H_ */
