/* sfm_b200.h -- C ABI of the B200-native matching + verification hot path.
 *
 * The reference (Justin-Huber/SfM-project) has no FFI: its boundary is the set of
 * module-level Python names that code/pipeline.py:1-3 star-imports.  The Python
 * drop-in modules under sfm-project_b200/ keep those names and call THIS library
 * through ctypes.  Each entry point below cites the reference interface it
 * replaces (paths relative to /root/reference).
 *
 * Conventions
 *   - plain pointers and sizes only; every device buffer is caller-owned
 *     (the Python host passes torch tensors' data_ptr()); the library allocates
 *     nothing on the device behind the caller's back.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *     the call returns without synchronising unless stated.
 *   - return value 0 = OK, negative = error; sfm_last_error() gives the text
 *     (thread-local).  Nothing throws across the boundary.
 *   - there is no CPU fallback: every entry point that computes needs a
 *     CUDA device of compute capability 10.0 (sm_100a code only).
 */
#ifndef SFM_B200_H
#define SFM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* every entry point below has default visibility; the rest of the library is hidden */
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define SFM_B200_ABI_VERSION 2   /* 2: sfm_match_knn2 lost its unused workspace arguments; sfm_peer_* and sfm_copy_async added */

/* error codes */
#define SFM_OK            0
#define SFM_ERR_ARG      -1   /* bad argument (null pointer, size out of range, misaligned) */
#define SFM_ERR_CUDA     -2   /* a CUDA runtime / driver call failed */
#define SFM_ERR_DEVICE   -3   /* no sm_100 device / wrong device */
#define SFM_ERR_STATE    -4   /* bank not filled, handle destroyed, ... */

/* descriptor metrics */
#define SFM_METRIC_L2       0  /* 128-byte uint8 descriptors, squared L2 (north-star SIFT workload) */
#define SFM_METRIC_HAMMING  1  /* 32-byte binary descriptors (the reference's literal ORB path)     */

/* ratio-test modes (SURVEY.md D8) */
#define SFM_RATIO_NONE      0  /* keep every query row that has a nearest neighbour            */
#define SFM_RATIO_CV2_F32   1  /* (double)sqrt_f32(D1) < ratio * (double)sqrt_f32(D2)          */
#define SFM_RATIO_EXACT_INT 2  /* D1 * den^2 < D2 * num^2 in int64                             */

/* matcher kernel selection */
#define SFM_MATCH_AUTO      0  /* tcgen05 kernel + exact refinement (default)   */
#define SFM_MATCH_TCGEN05   1
#define SFM_MATCH_SIMT      2  /* dp4a CUDA-core kernel (bring-up / cross-check) */

/* RANSAC options */
#define SFM_SOLVER_7PT 7
#define SFM_SOLVER_8PT 8
#define SFM_SCORE_SYM_EPIPOLAR 0   /* max(d1^2, d2^2) <= thr^2, cv2's FM_RANSAC metric */
#define SFM_SCORE_SAMPSON      1

const char* sfm_last_error(void);
int sfm_abi_version(void);

/* Device properties the host needs for grid sizing / diagnostics.
 * out[0]=SM count, out[1]=cc major, out[2]=cc minor, out[3]=max opt-in smem per block. */
int sfm_device_info(int device, int32_t out[4]);

/* ------------------------------------------------------------------ bank (K1)
 * Replaces the implicit hand-off "orb.detectAndCompute output -> bf.match input"
 * (code/feature_matching.py:44-50): descriptors are packed once, kept resident
 * in HBM, and every pair is matched from the bank.
 *
 * Storage layout inside the caller-provided buffer (all sections 1024-byte aligned):
 *   desc   int8  [n_images * feat_stride, 128]  L2: u8 ^ 0x80 (offset int8), zero padded rows
 *                                               Hamming: raw bytes, 32 used per row
 *   ext    int8  [n_images * feat_stride/128][2][128][16]  K-extension tile per 128 rows
 *                                               (encodes H0 - floor(|b|^2/2), see DESIGN.md)
 *   norm   int32 [n_images * feat_stride]       sum of squares of the offset-int8 row
 *   xy     float [n_images * feat_stride, 2]    keypoint pixel coordinates
 *   count  int32 [n_images]                     valid features per image
 * feat_stride = max_feats rounded up to 256.
 */
typedef struct sfm_bank sfm_bank_t;

int sfm_bank_storage_bytes(int max_images, int max_feats, int metric, size_t* out_bytes);
int sfm_bank_create(int device, int max_images, int max_feats, int metric,
                    void* storage, size_t storage_bytes, sfm_bank_t** out);
int sfm_bank_destroy(sfm_bank_t* bank);
/* feat_stride and byte offsets of the sections: out[0]=feat_stride, out[1..5]=desc,ext,norm,xy,count offsets */
int sfm_bank_layout(const sfm_bank_t* bank, int64_t out[6]);

/* Pack images [first_image, first_image+n_images) from DEVICE arrays:
 *   desc_u8 [n_images, src_stride, dim] (dim = 128 for L2, 32 for Hamming),
 *   counts  [n_images] (int32, device; may be NULL = all rows valid, n = src_stride),
 *   xy      [n_images, src_stride, 2] float32 (may be NULL).
 * One launch of the pack kernel for the whole batch. */
int sfm_bank_put_batch(sfm_bank_t* bank, int first_image, int n_images,
                       const uint8_t* desc_u8, int src_stride,
                       const int32_t* counts, const float* xy, void* stream);

/* After the storage has been filled by another rank's broadcast (no pack on this
 * rank), mark images [0,n_images) as present. */
int sfm_bank_mark_filled(sfm_bank_t* bank, int n_images);

/* --------------------------------------------------------------- matcher (K2)
 * Replaces, for the north-star SIFT/L2 workload, cv2.BFMatcher(NORM_L2).knnMatch(k=2)
 * + Lowe ratio (no call site in the reference; the literal call it displaces is
 * bf.match at code/feature_matching.py:50), for a whole list of image pairs
 * (the double loop of code/pipeline.py:38-41).
 *
 * knn_out int32 [n_pairs, feat_stride, 4] = (idx1, D1, idx2, D2) per query row of
 * image pairs[p][0] against the features of image pairs[p][1]; D are exact squared
 * L2 distances; ties go to the lowest train index; missing neighbours are -1.
 * Rows >= count[query image] are written as (-1,-1,-1,-1).
 * The kernels keep all scratch on chip: no workspace.
 */
typedef struct {
    int32_t impl;            /* SFM_MATCH_*                                                          */
    int32_t grid;            /* 0 = one CTA per SM                                                   */
    int32_t prefilter_mode;  /* SFM_RATIO_* (tcgen05 kernel only).  When non-zero, query rows that PROVABLY fail
                                this ratio test -- bounds from the sweep, see DESIGN.md -- are not refined and
                                read as (-1,-1,-1,-1); rows that can pass are exact as always, so
                                sfm_filter_matches* with the same test returns identical matches.  0 = every row. */
    int32_t sweep_only;      /* diagnostics: leave the sweep's candidate records in knn_out, skip refinement;
                                4 = the same without pre-filling knn_out (times the sweep kernel alone)          */
    double  prefilter_ratio; /* SFM_RATIO_CV2_F32: the ratio                                          */
    int32_t prefilter_num;   /* SFM_RATIO_EXACT_INT: ratio = num / den                                */
    int32_t prefilter_den;
} sfm_match_params;

int sfm_match_knn2(const sfm_bank_t* bank, const int32_t* pairs_dev, int n_pairs,
                   const sfm_match_params* params, int32_t* knn_out, void* stream);

/* Ratio test (+ optional mutual check) + ordered compaction + correspondence gather.
 * Replaces the Python post-filter at code/feature_matching.py:52-58 (there: sort +
 * absolute threshold; here: Lowe ratio in ascending queryIdx, the knnMatch idiom).
 *   knn_fwd  [n_pairs, feat_stride, 4]  query image -> train image
 *   knn_rev  same for the swapped pairs, or NULL when mutual == 0
 *   out_count int32 [n_pairs]            surviving matches per pair
 *   out_match int32 [n_pairs, cap, 3]    (queryIdx, trainIdx, D1), ascending queryIdx
 *   out_corr  float [n_pairs, cap, 4]    (x1,y1,x2,y2) pixel coordinates, may be NULL
 * cap = feat_stride.  One CTA per pair.
 */
typedef struct {
    int32_t ratio_mode;   /* SFM_RATIO_*            */
    int32_t mutual;       /* 0/1                    */
    double  ratio;        /* e.g. 0.75              */
    int64_t ratio_num;    /* exact_int: num/den     */
    int64_t ratio_den;
    int32_t max_distance_sq; /* keep only D1 < this (0 = off) */
    int32_t reserved[3];
} sfm_filter_params;

int sfm_filter_matches(const sfm_bank_t* bank, const int32_t* pairs_dev, int n_pairs,
                       const int32_t* knn_fwd, const int32_t* knn_rev,
                       const sfm_filter_params* params,
                       int32_t* out_count, int32_t* out_match, float* out_corr, void* stream);

/* Same filter, PACKED output (the layout the throughput path and the host copy use): pair p's matches are rows
 * [out_offset[p], out_offset[p+1]) of out_match / out_corr, so the whole result is one contiguous array of
 * out_offset[n_pairs] rows.
 *   out_count  int32 [n_pairs]       out_offset int32 [n_pairs + 1] (exclusive scan of out_count)
 *   out_match  int32 [>= total, 3]   out_corr   float [>= total, 4] or NULL
 * The caller sizes out_match / out_corr for the worst case n_pairs * feat_stride rows (or for a bound it knows).
 * Three launches: count, scan, write. */
int sfm_filter_matches_packed(const sfm_bank_t* bank, const int32_t* pairs_dev, int n_pairs,
                              const int32_t* knn_fwd, const int32_t* knn_rev,
                              const sfm_filter_params* params,
                              int32_t* out_count, int32_t* out_offset, int32_t* out_match, float* out_corr,
                              void* stream);

/* The matcher of the throughput path in one call: tcgen05 sweep -> exact refinement fused with this filter -> offsets ->
 * gather.  Output identical to sfm_match_knn2 + sfm_filter_matches_packed with the same parameters, but the 16-byte-per-row
 * kNN table is never materialised: the refinement applies the ratio test (and the mutual check against knn_rev, the finished
 * kNN table of the swapped pairs from sfm_match_knn2) to the top-2 it has just computed and keeps only the surviving rows.
 *   scratch   int32 [n_pairs, feat_stride, 4]   candidate records of the sweep, then the compacted rows per 256-row block
 *   blk_count int32 [n_pairs * feat_stride / 256]
 *   mp        may be NULL; a prefilter must use the filter's own ratio test (mode and ratio)
 * Four launches: sweep, refinement + filter, scan, gather. */
int sfm_match_pairs_packed(const sfm_bank_t* bank, const int32_t* pairs_dev, int n_pairs,
                           const sfm_match_params* mp, const sfm_filter_params* params, const int32_t* knn_rev,
                           int32_t* scratch, int32_t* blk_count,
                           int32_t* out_count, int32_t* out_offset, int32_t* out_match, float* out_corr,
                           void* stream);

/* The second half of sfm_match_pairs_packed on its own (refinement + filter, scan, gather): `scratch` holds the candidate
 * records of a sweep (sfm_match_knn2 with sweep_only = 4 and the filter's own prefilter).  Lets the caller run the NEXT
 * batch's sweep on one stream while this batch is refined and verified on another. */
int sfm_refine_filter_packed(const sfm_bank_t* bank, const int32_t* pairs_dev, int n_pairs,
                             const sfm_filter_params* params, const int32_t* knn_rev,
                             int32_t* scratch, int32_t* blk_count,
                             int32_t* out_count, int32_t* out_offset, int32_t* out_match, float* out_corr,
                             void* stream);

/* ----------------------------------------------------- Hamming matcher (K3)
 * Replaces cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=True).match followed by
 * sorted(key=distance) and the prefix `distance < 26`
 * (code/feature_matching.py:48-58) -- the reference's literal path.
 *   out_count int32 [n_pairs]
 *   out_match int32 [n_pairs, cap, 3]  (queryIdx, trainIdx, hamming), sorted by
 *             (distance asc, queryIdx asc), only distance < max_distance
 *   workspace device scratch of at least 2 * n_pairs * feat_stride * 8 bytes (the per-row nearest
 *             neighbours of both directions, read by the cross-check); caller-owned like every buffer
 */
int sfm_match_hamming(const sfm_bank_t* bank, const int32_t* pairs_dev, int n_pairs,
                      int max_distance, int32_t* out_count, int32_t* out_match,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------ RANSAC-F (K4)
 * Fills the empty code/geometric_verification.py (0 bytes; placeholder comment
 * at code/pipeline.py:60).  Conventions follow cv2.findFundamentalMat(FM_RANSAC):
 * F is 3x3 row-major double with x2^T F x1 = 0, scaled so F[8] == 1 when
 * |F[8]| > FLT_EPSILON; mask is uint8 per correspondence.
 *
 *   corr    float [n_pairs, corr_stride, 4]  (x1,y1,x2,y2)
 *   count   int32 [n_pairs]                  correspondences per pair (<= corr_stride)
 *   pair_id uint32[n_pairs] or NULL          RNG stream id of each pair (NULL = index)
 *   samples uint32[max_iters, 8] or NULL     explicit minimal samples (shared by all pairs)
 *   out_F      double [n_pairs, 9]
 *   out_ninl   int32  [n_pairs]   (0 = no model)
 *   out_mask   uint8  [n_pairs, corr_stride]
 *   out_iters  int32  [n_pairs]   hypotheses actually evaluated (may be NULL)
 */
typedef struct {
    int32_t solver;       /* SFM_SOLVER_7PT / SFM_SOLVER_8PT          */
    int32_t score;        /* SFM_SCORE_*                               */
    float   threshold;    /* pixels                                    */
    int32_t max_iters;    /* hypothesis budget per pair                */
    double  confidence;   /* adaptive stop; >= 1.0 disables it         */
    uint64_t seed;
    int32_t lo_refit;     /* 0/1: normalised 8-point refit on inliers  */
    int32_t min_inliers;  /* pairs below this report n_inl=0 (0 = off) */
    int32_t reserved[4];
} sfm_ransac_params;

int sfm_ransac_f_batch(const float* corr, int corr_stride, const int32_t* count, int n_pairs,
                       const uint32_t* pair_id, const uint32_t* samples,
                       const sfm_ransac_params* params,
                       double* out_F, int32_t* out_ninl, uint8_t* out_mask, int32_t* out_iters,
                       void* stream);

/* Packed layout (pairs back to back, as written by sfm_filter_matches_packed):
 *   corr     float [total, 4]        offsets int32 [n_pairs + 1]
 *   out_mask uint8 [total]           max_count = upper bound of any pair's correspondence count (e.g. feat_stride)
 * Results are identical to the strided call on the same correspondences. */
int sfm_ransac_f_packed(const float* corr, const int32_t* offsets, int n_pairs, int max_count,
                        const uint32_t* pair_id, const uint32_t* samples,
                        const sfm_ransac_params* params,
                        double* out_F, int32_t* out_ninl, uint8_t* out_mask, int32_t* out_iters,
                        void* stream);

/* ---------------------------------------------------- RANSAC-H (SURVEY.md 8f rank 2)
 * Second model of the verification stage the reference left empty
 * (code/geometric_verification.py, 0 bytes; code/pipeline.py:60-65): a planar or
 * purely rotating pair is explained by a homography, and the H-vs-F inlier
 * ratio classifies the pair for the scene graph.  Conventions follow
 * cv2.findHomography(RANSAC): x2 ~ H x1, H is 3x3 row-major double scaled so
 * H[8] == 1, inlier iff |proj(H x1) - x2|^2 <= thr^2.  Buffers, sampling
 * (seed / pair_id / explicit samples: the first 4 of each row of 8) and the
 * adaptive stop are exactly those of sfm_ransac_f_*; params->solver and
 * params->score are ignored (4-point DLT, forward transfer error).
 *   stop_target int32 [n_pairs] or NULL   when the caller only needs to know whether H can reach that many inliers
 *                                          (the scene-graph test n_H > r * n_F), sampling stops as soon as a model with
 *                                          max(best so far, target) inliers would have been found with params->confidence:
 *                                          a general (non-planar) pair then costs 32 hypotheses instead of max_iters.
 */
int sfm_ransac_h_batch(const float* corr, int corr_stride, const int32_t* count, int n_pairs,
                       const uint32_t* pair_id, const uint32_t* samples, const int32_t* stop_target,
                       const sfm_ransac_params* params,
                       double* out_H, int32_t* out_ninl, uint8_t* out_mask, int32_t* out_iters,
                       void* stream);
int sfm_ransac_h_packed(const float* corr, const int32_t* offsets, int n_pairs, int max_count,
                        const uint32_t* pair_id, const uint32_t* samples, const int32_t* stop_target,
                        const sfm_ransac_params* params,
                        double* out_H, int32_t* out_ninl, uint8_t* out_mask, int32_t* out_iters,
                        void* stream);

/* --------------------------------------- two-view initialisation (SURVEY.md 8f rank 4)
 * The consumer of (F, inlier mask): feeds the reference's empty
 * code/3d_reconstruction.py (0 bytes; imported at code/pipeline.py:4).  Per pair:
 * E = K2^T F K1 (unit Frobenius norm), its four (R, t) decompositions, the
 * cheirality vote by DLT triangulation of the inlier correspondences, and the
 * points of the winner.  Conventions follow cv2.recoverPose(E, pts1, pts2, K,
 * distanceThresh) + cv2.triangulatePoints: x2 ~ R x1 + t, |t| = 1, candidate
 * order (R1,t) (R2,t) (R1,-t) (R2,-t) with ties to the earlier one; a point
 * votes iff its depth lies in (0, distance_thresh) in both cameras.
 *
 *   corr / count / offsets   as for sfm_ransac_f_batch / _packed
 *   in_mask  uint8  [rows] or NULL   correspondences to use (the RANSAC-F inlier mask)
 *   F        double [n_pairs, 9]     all-zero rows (no model) give an all-zero result
 *   cam      double [n_pairs, 8]     fx1 fy1 cx1 cy1 fx2 fy2 cx2 cy2 (pinhole, zero skew)
 *   out_R    double [n_pairs, 9]     out_t double [n_pairs, 3]
 *   out_E    double [n_pairs, 9] or NULL
 *   out_ngood int32 [n_pairs]        votes of the chosen candidate (0 = no pose)
 *   out_mask uint8  [rows]           in_mask AND positive bounded depth in both cameras
 *   out_X    float  [rows, 3] or NULL   triangulated points, camera-1 frame (zeros where out_mask is 0)
 */
int sfm_two_view_pose_batch(const float* corr, int corr_stride, const int32_t* count, int n_pairs,
                            const uint8_t* in_mask, const double* F, const double* cam, double distance_thresh,
                            double* out_R, double* out_t, double* out_E, int32_t* out_ngood,
                            uint8_t* out_mask, float* out_X, void* stream);
int sfm_two_view_pose_packed(const float* corr, const int32_t* offsets, int n_pairs,
                             const uint8_t* in_mask, const double* F, const double* cam, double distance_thresh,
                             double* out_R, double* out_t, double* out_E, int32_t* out_ngood,
                             uint8_t* out_mask, float* out_X, void* stream);

/* ------------------------------------------------- ORB descriptor stage (SURVEY.md 8f rank 1, stage 1)
 * The descriptor half of `orb.detectAndCompute(gray, None)` (code/feature_matching.py:42-45) for keypoints cv2 detected:
 * image pyramid, per-level Gaussian blur, rotated rBRIEF tests -- each bit-exact against cv2 4.13.  The host computes
 * the level sizes, the 8.8 fixed-point resize tables and each keypoint's rounded level position and (cos, sin); the
 * descriptors (32 bytes each) can be written straight into a Hamming bank's rows (out_stride = 32).
 *   sfm_orb_resize   INTER_LINEAR_EXACT of a uint8 image; xtab / ytab int32 [dw, 2] / [dh, 2] = (source index, weight of
 *                    the next source pixel in 1/256) per destination column / row
 *   sfm_orb_blur     GaussianBlur(7 x 7, sigma 2, BORDER_REFLECT_101) as cv2 computes it for ORB (float32 sepFilter2D)
 *   sfm_orb_describe level_ptr / level_pitch are HOST arrays of device pointers / pitches of the BLURRED levels;
 *                    kp int32 [n, 4] = (x, y in the level image, level, 0), rot float [n, 2] = (cos, sin) of the angle
 */
int sfm_orb_resize(const uint8_t* src, int sw, int sh, int spitch, uint8_t* dst, int dw, int dh, int dpitch,
                   const int32_t* xtab, const int32_t* ytab, void* stream);
int sfm_orb_blur(const uint8_t* src, int w, int h, int spitch, uint8_t* dst, int dpitch, void* stream);
int sfm_orb_describe(const uint8_t* const* level_ptr, const int32_t* level_pitch, int n_levels,
                     const int32_t* kp, const float* rot, int n_keypoints,
                     uint8_t* out_desc, int out_stride, void* stream);

/* Stage 2: the keypoint half of `orb.detectAndCompute` (code/feature_matching.py:44-45), per pyramid level, bit-exact
 * against cv2.ORB_create().detect including the ORDER of the keypoints.
 *   sfm_orb_fast_detect   FAST-9/16 corner scores (uint8 [h, w], 0 = no corner at `threshold`), 3 x 3 non-maximum
 *                         suppression, `border` rule, row-major compaction: out_xy int32 [n, 2], out_resp float [n]
 *                         (the FAST score), *total = n.  Size out_xy / out_resp for w * h / 4 keypoints (the most 3 x 3
 *                         suppression can leave); row_count is int32 [h] scratch.  Three launches.
 *   sfm_orb_retain_best   HOST function: KeyPointsFilter::retainBest on host responses -- the indices of the keypoints whose
 *                         response reaches the n_points-th largest, in the order libstdc++'s nth_element + partition leave
 *                         them (that order is the order of cv2's keypoints).  Returns the number kept.
 *   sfm_orb_harris_angle  Harris response (7 x 7, k = 0.04) and intensity-centroid orientation (degrees, cv::fastAtan2) of
 *                         the candidates sel[0..n) (indices into xy; NULL = the first n) on the UNBLURRED level.
 */
int sfm_orb_fast_detect(const uint8_t* img, int w, int h, int pitch, int threshold, int border,
                        uint8_t* score, int32_t* row_count, int32_t* total, int32_t* out_xy, float* out_resp, void* stream);
int sfm_orb_retain_best(const float* response_host, int n, int n_points, int32_t* out_index);
int sfm_orb_harris_angle(const uint8_t* img, int w, int h, int pitch, const int32_t* xy, const int32_t* sel, int n,
                         int32_t* out_xy, float* out_resp, float* out_angle, void* stream);

/* ------------------------------------------------------------- feature tracks (f5)
 * The output of correspondence search (Schoenberger & Frahm 2016, §2.1) that registration and multi-view triangulation
 * read: the reference's empty code/3d_reconstruction.py (imported at code/pipeline.py:4) would build it from the
 * `pair_matches` list of code/pipeline.py:43-47.  A track is a connected component of the graph whose nodes are
 * n = image * S + feature (S = features per image, n_images * S < 2^31) and whose edges are the used match rows.
 *
 *   pairs      int32 [n_pairs, 2]   (i, j) per pair
 *   row_start  int64 [n_pairs]      pair p owns rows [row_start[p], row_start[p] + n_rows[p]) of rows / row_flag
 *   n_rows     int32 [n_pairs]
 *   rows       int32 [., 3]         (q, t, d2): the edge (i*S + q, j*S + t); d2 is not read
 *   row_flag   uint8 [.] or NULL    a row is used only when its flag is non-zero (NULL = every row)
 *   n_inliers  int32 [n_pairs] or NULL   pairs with n_inliers[p] < params->min_pair_inliers contribute no row
 * A row that would be used but has q or t outside [0, S) (or whose pair names an image outside [0, n_images)) is counted in
 * counts[4] and not used.
 *
 * Candidates are the connected components of the used edges.  A candidate holding two features of one image is
 * conflicting (counts[2]) and dropped unless keep_conflicts; then a candidate of fewer than min_length observations is
 * dropped (counts[3]).  Kept tracks are numbered in ascending order of their smallest node, observations ascend by node:
 * the output depends only on the SET of used edges (not on row / pair order, duplicates or both-direction rows).
 *
 *   sfm_tracks_workspace_bytes  size of the caller-owned device workspace (256-byte aligned)
 *   sfm_tracks_init             start a job (one launch)
 *   sfm_tracks_hook             add the used rows of a batch of pairs (one launch; any number of calls per job)
 *   sfm_tracks_finalize         write the tracks (14 launches; the state stays valid for more hooks and another finalize):
 *       track_of int32 [n_images, S]        track id of every feature, -1 = none
 *       offsets  int64 [>= n_nodes/2 + 1]   track k owns observations [offsets[k], offsets[k+1])
 *       obs      int32 [>= n_nodes, 2]      (image, feature)
 *       counts   int64 [5]                  tracks, observations, conflicting candidates, short candidates, invalid rows
 *     The buffers are sized for the worst case, so nothing waits for the host.
 */
typedef struct {
    int32_t min_pair_inliers;  /* see n_inliers above                             */
    int32_t min_length;        /* >= 2                                            */
    int32_t keep_conflicts;    /* 0/1                                             */
    int32_t reserved[5];
} sfm_track_params;

int sfm_tracks_workspace_bytes(int n_images, int S, size_t* out_bytes);
int sfm_tracks_init(int n_images, int S, void* workspace, size_t workspace_bytes, void* stream);
int sfm_tracks_hook(int n_images, int S, const int32_t* pairs, int n_pairs, const int64_t* row_start, const int32_t* n_rows,
                    const int32_t* rows, const uint8_t* row_flag, const int32_t* n_inliers, const sfm_track_params* params,
                    void* workspace, size_t workspace_bytes, void* stream);
int sfm_tracks_finalize(int n_images, int S, const sfm_track_params* params, void* workspace, size_t workspace_bytes,
                        int32_t* track_of, int64_t* offsets, int32_t* obs, int64_t* counts, void* stream);

/* ------------------------------------------------------------ track triangulation
 * One 3-D point per feature track from known cameras: what known-pose reconstruction (calibrated rigs, poses from GPS /
 * IMU) computes, and what incremental registration calls after every image it adds.  Cameras follow x ~ K (R X + t),
 * X in world coordinates (the two-view step's frame when camera 1 is [I|0]).
 *
 *   offsets, obs, track_counts   the tracks exactly as sfm_tracks_finalize writes them; the track count is read from
 *                                track_counts[0] on the device, clamped to max_tracks (the capacity of offsets - 1 and of
 *                                the per-track outputs), so nothing waits for the host
 *   xy         float  [n_images, xy_stride, 2]   keypoint pixel coordinates (a bank's xy section); S <= xy_stride
 *   cams       double [n_images, 16]             fx fy cx cy, R (row-major), t
 *   registered uint8  [n_images] or NULL         observations in images with registered[i] == 0 are not used (NULL = all)
 *
 * Per track k, over its M usable observations (registered images, in obs order), all in fp64:
 *   normalised coordinates  x^ = ((double)x - cx) / fx, y^ = ((double)y - cy) / fy
 *   DLT rows                (x^ r3 - r1) * fx and (y^ r3 - r2) * fy of [R|t], added serially in row order to the 4 x 4
 *                           normal matrix; the point is its eigenvector of the smallest eigenvalue (6 cyclic Jacobi
 *                           sweeps), divided by w when |w| > 1e-300.  The focal lengths make each row a pixel residual
 *                           times the depth, so the views of different cameras weigh alike
 *   reprojection            p = R X + t; the squared error is ((p0 * (1/p2) - x^) * fx)^2 + ((p1 * (1/p2) - y^) * fy)^2;
 *                           an observation is an inlier iff p2 > 0 and that error <= max_error^2
 *   hypotheses              the DLT of observations draw_sample(seed, k, h, 2, M) (the RANSAC kernels' sampler; rows of
 *                           the earlier observation first), kept iff both depths are > 0 and the cosine of the angle
 *                           between X - C_a and X - C_b (C = -R^T t) is <= cos(min_angle).  Batches of 32, 32, 64, 128, ...
 *                           hypotheses, the RANSAC stop rule after each batch, at most max_iters; a hypothesis replaces
 *                           the best only with strictly more inliers
 *   refit                   at most 2 rounds of the N-view DLT over the current inliers; kept iff it has at least as many
 *   status                  0 triangulated, 1 too few views (M < 2), 2 no hypothesis kept, 3 fewer than min_inliers
 *                           inliers, 4 an observation names an image outside [0, n_images) or a feature outside [0, S)
 *                           (the track is counted and none of its coordinates are read)
 * Outputs:
 *   out_X           double [max_tracks, 3]   zeros unless status 0
 *   out_n_inliers   int32  [max_tracks]      inliers of the final point (status 0 and 3), else 0
 *   out_status      uint8  [max_tracks]
 *   out_obs_inlier  uint8  [obs]             per observation, in obs order (0 unless status 0)
 *   out_obs_error   float  [obs]             pixel reprojection error of the final point; +inf behind the camera, NaN in
 *                                            unregistered images and for tracks without a point.  The kernel also uses a
 *                                            track's slice as scratch for observations beyond the shared-memory stage
 *   out_counts      int64  [5]               tracks per status
 * Bit-identical to oracle/triangulate.c.  One launch (after a memset of out_counts).
 */
typedef struct {
    double   max_error;    /* pixels, > 0 (COLMAP's mapper filter default: 4)         */
    double   min_angle;    /* degrees, in [0, 90) (COLMAP's default: 1.5)             */
    double   confidence;   /* adaptive stop; >= 1.0 disables it                        */
    uint64_t seed;
    int32_t  max_iters;    /* hypothesis budget per track, > 0                         */
    int32_t  min_inliers;  /* >= 2                                                     */
    int32_t  reserved[6];
} sfm_triangulate_params;

int sfm_triangulate_tracks(int n_images, int S, const int64_t* offsets, const int32_t* obs, const int64_t* track_counts,
                           int64_t max_tracks, const float* xy, int xy_stride, const double* cams, const uint8_t* registered,
                           const sfm_triangulate_params* params, double* out_X, int32_t* out_n_inliers, uint8_t* out_status,
                           uint8_t* out_obs_inlier, float* out_obs_error, int64_t* out_counts, void* stream);

/* ------------------------------------------------------------ absolute pose / registration
 * A camera pose from 2-D / 3-D correspondences: the step of incremental reconstruction that registers a new image against
 * the points triangulated so far.  Cameras follow x ~ K (R X + t), as in track triangulation.
 *
 * sfm_pnp_gather: the correspondences of n_query images.  For query q, they are the features f of image[q] (f ascending)
 * whose track k = track_of[image[q] * S + f] satisfies 0 <= k < min(track_counts[0], max_tracks) and point_status[k] == 0:
 *   track_of, track_counts   as sfm_tracks_finalize writes them (the track count is read on the device)
 *   point_status, X          uint8 [max_tracks], double [max_tracks, 3]: as sfm_triangulate_tracks writes them
 *   xy                       float [n_images, xy_stride, 2]   keypoint pixel coordinates; S <= xy_stride
 * Outputs in the strided layout of sfm_pnp_ransac with stride S (query q owns entries [q * S, q * S + out_count[q])):
 *   out_xy float [n_query, S, 2], out_X double [n_query, S, 3], out_feature int32 [n_query, S], out_count int32 [n_query].
 * An image outside [0, n_images) gets out_count 0.  Entries past out_count[q] are not written.  One launch.
 *
 * sfm_pnp_ransac: one pose per query from the first count[q] (clamped to stride) correspondences of query q:
 *   cams    double [n_images, 16]   fx fy cx cy ... (the table track triangulation reads); row image[q] gives the intrinsics
 *   xy      float  [n_query, stride, 2]   pixel coordinates;  X  double [n_query, stride, 3]   world points
 * All in fp64 with IEEE basic operations and sqrt only:
 *   normalised coordinates  x^ = ((double)x - cx) / fx, y^ = ((double)y - cy) / fy
 *   inlier                  p = R X + t, p2 > 0 and ((p0 * (1/p2) - x^) * fx)^2 + ((p1 * (1/p2) - y^) * fy)^2 <= max_error^2
 *                           (track triangulation's predicate, so a pose and a point agree on what an inlier is)
 *   hypotheses              the correspondences draw_sample(seed, image[q], h, 3, M) (the RANSAC kernels' sampler; the
 *                           image id is the stream id, so a query's bits do not depend on its batch), solved by Lambda Twist
 *                           P3P (Persson & Nordberg, ECCV 2018): the cubic's root by Newton iterations, the 3 x 3 symmetric
 *                           eigenproblem by 8 cyclic Jacobi sweeps, at most 5 Gauss-Newton steps on the depths, R from a
 *                           3 x 3 inverse; up to 4 poses per sample in a fixed root order, a root dropped when a depth is
 *                           not > 0 or R, t is not finite.  Batches of 32, 32, 64, 128, ... hypotheses, the RANSAC stop rule
 *                           (m = 3) after each, at most max_iters; a pose replaces the best only with strictly more inliers,
 *                           in (hypothesis, root) order
 *   refinement              when refine_iters > 0, at most 2 rounds while the pose has >= 3 inliers: at most refine_iters
 *                           Gauss-Newton steps on the pixel residuals of the round's inliers (sums over 256 lanes, each lane
 *                           in correspondence order, then a fixed tree; the 6 x 6 normal equations by Cholesky), perturbing
 *                           the pose in the camera frame: R' = dR R, t' = dR t + dt with dR the normalised quaternion
 *                           (1, w/2) and the Jacobian taken at p = R X + t, so the step's linearisation error scales with
 *                           the depth and not with |X| (worlds far from their origin refine as well as centred ones); a
 *                           step taken only if the cost drops; the round's pose is kept iff it moved and has at least as
 *                           many inliers
 *   status                  0 registered, 1 fewer than 3 correspondences, 2 no pose from any sample, 3 fewer inliers than
 *                           min_inliers or min_inlier_ratio * M, 4 image outside [0, n_images) or a focal length that is not
 *                           positive and finite (the query is counted and none of its correspondences are read)
 * Outputs:
 *   out_pose       double [n_query, 12]      R (row-major), t: drops into cams[image, 4:]; zeros unless status 0
 *   out_n_inliers  int32  [n_query]          inliers of the final pose (status 0 and 3), else 0
 *   out_status     uint8  [n_query]
 *   out_mask       uint8  [n_query, stride]  inlier flags of the final pose (0 unless status 0); used as scratch
 *   out_iters      int32  [n_query] or NULL  hypotheses drawn
 *   out_counts     int64  [5]                queries per status
 * Bit-identical to oracle/pnp.c.  One launch (after a memset of out_counts).
 */
typedef struct {
    double   max_error;         /* pixels, > 0 (COLMAP's IncrementalMapper abs_pose_max_error: 12)                 */
    double   confidence;        /* adaptive stop; >= 1.0 disables it                                               */
    uint64_t seed;
    int32_t  max_iters;         /* hypothesis budget per query, > 0                                                */
    int32_t  min_inliers;       /* >= 3 (COLMAP's abs_pose_min_num_inliers: 30)                                    */
    double   min_inlier_ratio;  /* in [0, 1] (COLMAP's abs_pose_min_inlier_ratio: 0.25)                            */
    int32_t  refine_iters;      /* Gauss-Newton steps per refinement round, in [0, 1000]; 0 = no refinement        */
    int32_t  reserved[5];
} sfm_pnp_params;

int sfm_pnp_gather(int n_images, int S, const int32_t* track_of, const int64_t* track_counts, int64_t max_tracks,
                   const uint8_t* point_status, const double* X, const float* xy, int xy_stride, const int32_t* image, int n_query,
                   float* out_xy, double* out_X, int32_t* out_feature, int32_t* out_count, void* stream);
int sfm_pnp_ransac(int n_images, const double* cams, const int32_t* image, int n_query, const float* xy, const double* X, int stride,
                   const int32_t* count, const sfm_pnp_params* params, double* out_pose, int32_t* out_n_inliers, uint8_t* out_status,
                   uint8_t* out_mask, int32_t* out_iters, int64_t* out_counts, void* stream);

/* ------------------------------------------------------------ bundle adjustment
 * Every registered camera and every triangulated point refined together: the step that makes incremental reconstruction
 * more than a first guess.  Cameras follow x ~ K (R X + t), as in track triangulation; the intrinsics stay fixed.
 *
 *   offsets, obs, track_counts   the tracks as sfm_tracks_finalize writes them (the track count is read from track_counts[0]
 *                                on the device, clamped to max_tracks; the observation count is offsets[n_tracks], clamped to
 *                                max_obs), so nothing waits for the host
 *   point_status, obs_inlier, X  uint8 [max_tracks], uint8 [max_obs], double [max_tracks, 3]: as sfm_triangulate_tracks writes them
 *   xy         float  [n_images, xy_stride, 2]   keypoint pixel coordinates; S <= xy_stride
 *   cams       double [n_images, 16]             fx fy cx cy, R (row-major), t
 *   registered uint8  [n_images] or NULL         NULL = every image
 *   fixed      uint8  [n_images] or NULL         poses held fixed; NULL = the lowest-index registered image (the gauge's
 *                                                rotation and origin; the scale is left to the damping)
 *
 * An observation is used iff its track has point status 0, its obs_inlier is 1 and its image is registered.  A camera is
 * variable iff it is registered, not fixed and has a used observation; a point is adjusted iff it has 2 or more used
 * observations.  Every other pose and point is returned bit-identical to its input.
 * The cost is the sum over the used observations of ((p0 * (1/p2) - x^) * fx)^2 + ((p1 * (1/p2) - y^) * fy)^2 with
 * p = R X + t and x^ = ((double)x - cx) / fx (track triangulation's residual), plain squares.  Levenberg-Marquardt in fp64:
 *   parameters   a camera moves by registration's camera-frame perturbation R' = dR(w) R, t' = dR(w) t + dt (dR the
 *                normalised quaternion (1, w/2), the Jacobian taken at p), a point by X' = X + dX
 *   step         the damped normal equations (H + lambda diag(H)) [dc; dX] = -J^T r reduced to the variable cameras by the
 *                Schur complement S = U - W V^-1 W^T (cameras compacted to 0..Nv-1, S dense, Nv <= 1024), solved by a blocked
 *                Cholesky, then the points back-substituted; a trial with any used observation at p2 <= 0, or whose system
 *                is not positive definite, is rejected
 *   lambda       starts at 1e-4; Nielsen's rule: accepted (cost drops): lambda *= max(1/3, 1 - (2 rho - 1)^3), nu = 2;
 *                rejected: lambda *= nu, nu *= 2.  The Jacobians are recomputed only after an accepted step
 *   summary.status  0 function_tolerance: an accepted step lowered the cost by less than function_tolerance * cost
 *                   1 parameter_tolerance: an accepted step had |dx| <= parameter_tolerance * (|x| + parameter_tolerance),
 *                     x = (t of the variable cameras, the adjusted points), dx = (w, dt, dX)
 *                   2 max_iterations: max_iters trials (rejected ones count)
 *                   3 no_progress: lambda passed 1e32; the last accepted state is returned
 *                   4 nothing_to_adjust: no variable camera and no adjusted point
 *                   5 invalid: a used observation's track names an image outside [0, n_images) or a feature outside [0, S),
 *                     or a registered image with used observations has a focal length that is not positive and finite
 * Every sum runs in a fixed order (no floating-point atomics), so the result is bit-identical from run to run, on any
 * stream, and with unregistered images added (the layout of the reduced system depends only on Nv).
 * Outputs:
 *   out_pose       double [n_images, 12]   R (row-major), t: drops into cams[:, 4:]
 *   out_X          double [max_tracks, 3]
 *   out_obs_error  float  [obs]            pixel reprojection error after the adjustment, as sfm_triangulate_tracks defines it
 *                                          (+inf behind the camera, NaN in unregistered images and for tracks without a point)
 *   out_summary    sfm_bundle_summary      (device memory)
 * sfm_bundle_workspace_bytes sizes the caller-owned device workspace (the reduced system alone takes (6 n_images)^2 doubles);
 * n_images is at most 1024.  The call issues 4 + 5 * max_iters launches whatever the data: once the solve has stopped, the
 * remaining iterations' kernels exit at once.
 */
typedef struct {
    double   function_tolerance;   /* >= 0 (default 1e-6)                          */
    double   parameter_tolerance;  /* >= 0 (default 1e-8)                          */
    int32_t  max_iters;            /* trials, in [1, 10000] (default 50)           */
    int32_t  reserved[11];
} sfm_bundle_params;

typedef struct {
    int64_t  status;               /* see above                                    */
    int64_t  iterations;           /* trials run                                   */
    int64_t  accepted;             /* accepted steps                               */
    int64_t  used_obs;
    int64_t  variable_cameras;     /* Nv                                           */
    int64_t  adjusted_points;
    double   initial_cost;
    double   final_cost;
} sfm_bundle_summary;

int sfm_bundle_workspace_bytes(int n_images, int64_t max_tracks, int64_t max_obs, size_t* out_bytes);
int sfm_bundle_adjust(int n_images, int S, const int64_t* offsets, const int32_t* obs, const int64_t* track_counts, int64_t max_tracks,
                      int64_t max_obs, const uint8_t* point_status, const uint8_t* obs_inlier, const double* X, const float* xy,
                      int xy_stride, const double* cams, const uint8_t* registered, const uint8_t* fixed, const sfm_bundle_params* params,
                      void* workspace, size_t workspace_bytes, double* out_pose, double* out_X, float* out_obs_error,
                      sfm_bundle_summary* out_summary, void* stream);

/* ------------------------------------------ result regions in peer memory (multi-GPU gather)
 * Across ranks, the reference's `pair_matches.append(Pair(...))` (code/pipeline.py:43-47) becomes: every rank
 * writes the packed match rows / inlier flags of its pair block straight into a region of the gathering rank's
 * HBM over NVLink (copy engines, no SMs, no staging, no padded collective).  The gathering rank allocates the
 * region and exports a 64-byte handle (cudaIpcMemHandle_t); the other processes of the box open it and use
 * sfm_copy_async with the mapped pointer as destination.  These four calls are the only place where the library
 * owns device memory.
 *   sfm_peer_alloc  allocate `bytes` on `device` (256-byte aligned), return the pointer and its handle
 *   sfm_peer_open   map another process's region into this process (peer access is enabled on first use; SFM_ERR_DEVICE when
 *                   the two GPUs have no direct peer path -- the caller then uses send/recv instead)
 *   sfm_peer_close  unmap a region obtained from sfm_peer_open
 *   sfm_peer_free   free a region obtained from sfm_peer_alloc
 *   sfm_copy_async  cudaMemcpyAsync(dst, src, bytes) on `stream`; either side may be local, peer or pinned host
 */
int sfm_peer_alloc(int device, size_t bytes, void** out_ptr, uint8_t out_handle[64]);
int sfm_peer_open(int device, const uint8_t handle[64], void** out_ptr);
int sfm_peer_close(int device, void* ptr);
int sfm_peer_free(int device, void* ptr);
int sfm_copy_async(void* dst, const void* src, size_t bytes, void* stream);

/* -------------------------------------------------------------- diagnostics
 * Issue `n_tiles` 128x128x160 int8 tcgen05 MMAs per CTA with no epilogue: the
 * attainable tensor-pipe rate the matcher is measured against (MEASURED_PEAKS.json
 * has no int8 entry).  out_ms receives the kernel time measured with CUDA events
 * (this call synchronises). */
int sfm_probe_int8_mma(int device, int n_tiles, float* out_ms, double* out_ops);

/* Bring-up aid used by tests: run the tcgen05 matcher on ONE pair (pairs_dev[0..1]) with a single CTA and
 * dump the raw int32 accumulators of the first unit / first train tile (acc_out int32 [256,128]).
 * mode 0 = descriptor MMAs + K-extension MMA, 1 = descriptor MMAs only, 2 = K-extension only.
 * knn_out int32 [feat_stride, 4]. */
int sfm_debug_tc_tile(const sfm_bank_t* bank, const int32_t* pairs_dev, int mode, int32_t* knn_out,
                      int32_t* acc_out, void* stream);

/* Diagnostics of the exact-refinement kernel: enable != 0 switches the counters on for later launches;
 * out[0] = query rows that needed the whole-image brute force, out[1] = candidate distances recomputed. */
int sfm_debug_refine_stats(int enable, int64_t out[2]);

/* Counters of kernels launched by this library since load (per process). */
int64_t sfm_launch_count(void);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* SFM_B200_H */
