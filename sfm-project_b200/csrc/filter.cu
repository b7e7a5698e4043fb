// filter.cu -- Lowe ratio test (+ mutual check) + ordered compaction + correspondence gather (K5).
//
// Replaces the per-pair Python post-filter of the reference (code/feature_matching.py:52-58: sort by
// distance and keep the prefix < 26) for the north-star L2 path: the knnMatch idiom
// `m.distance < ratio * n.distance`, evaluated bit-exactly (SURVEY.md D8), emitted in ascending
// queryIdx like cv2's knnMatch, plus the pixel coordinates RANSAC consumes.
#include "match_common.cuh"

namespace sfm {

// One CTA per pair, rows visited in order so the output is sorted by queryIdx.
//   kWrite == false : count the surviving rows only (first pass of the packed layout)
//   kWrite == true  : write (queryIdx, trainIdx, D1) and the correspondence (x1,y1,x2,y2) of every surviving row at
//                     out_base[p] + rank, where out_base is NULL for the strided layout (base = p * feat_stride)
#ifndef SFM_FILTER_ROWS
#define SFM_FILTER_ROWS 4
#endif
template <bool kWrite>
__global__ void __launch_bounds__(256) filter_kernel(
    const int32_t* __restrict__ pairs, const int32_t* __restrict__ count, const float* __restrict__ xy, int feat_stride,
    const int32_t* __restrict__ knn_fwd, const int32_t* __restrict__ knn_rev, int mode, int mutual, double ratio,
    long long num2, long long den2, int max_d, int32_t* __restrict__ out_count, const int32_t* __restrict__ out_base,
    int32_t* __restrict__ out_match, float* __restrict__ out_corr)
{
    __shared__ int warp_tot[8];
    __shared__ int base;
    const int p = blockIdx.x;
    const int img_q = pairs[2 * p], img_t = pairs[2 * p + 1];
    const int nq = count[img_q];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    const int4* fwd = reinterpret_cast<const int4*>(knn_fwd) + (long long)p * feat_stride;
    const int4* rev = knn_rev ? reinterpret_cast<const int4*>(knn_rev) + (long long)p * feat_stride : nullptr;
    const long long obase = kWrite ? (out_base ? (long long)out_base[p] : (long long)p * feat_stride) : 0;
    // every thread owns kRows consecutive rows of a 1024-row slab: four 16-byte loads in flight per thread, one barrier round
    // per slab; ranks follow (thread, j) = ascending row order
    constexpr int kRows = SFM_FILTER_ROWS;
    for (int r0 = 0; r0 < nq; r0 += 256 * kRows) {
        const int rt = r0 + threadIdx.x * kRows;
        int4 k[kRows];
        bool keep[kRows];
#pragma unroll
        for (int j = 0; j < kRows; ++j) k[j] = (rt + j < nq) ? fwd[rt + j] : make_int4(-1, -1, -1, -1);
        int cnt = 0;
#pragma unroll
        for (int j = 0; j < kRows; ++j) {
            bool kp = k[j].x >= 0 && ratio_keep(k[j].y, k[j].w, mode, ratio, num2, den2);
            if (kp && max_d > 0) kp = k[j].y < max_d;
            if (kp && mutual) kp = rev[k[j].x].x == rt + j;
            keep[j] = kp;
            cnt += kp;
        }
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        if (kWrite && cnt) {
            int off = base + incl - cnt;
            for (int w = 0; w < warp; ++w) off += warp_tot[w];
#pragma unroll
            for (int j = 0; j < kRows; ++j) {
                if (!keep[j]) continue;
                const long long o = obase + off++;
                out_match[o * 3 + 0] = rt + j;
                out_match[o * 3 + 1] = k[j].x;
                out_match[o * 3 + 2] = k[j].y;
                if (out_corr) {
                    const float2 a = reinterpret_cast<const float2*>(xy)[(long long)img_q * feat_stride + rt + j];
                    const float2 b = reinterpret_cast<const float2*>(xy)[(long long)img_t * feat_stride + k[j].x];
                    reinterpret_cast<float4*>(out_corr)[o] = make_float4(a.x, a.y, b.x, b.y);
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int w = 0; w < 8; ++w) tot += warp_tot[w];
            base += tot;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0 && out_count) out_count[p] = base;
}

// Exclusive scan of the per-pair counts (one CTA; P is a few thousand at most per batch): offset[0..P].
__global__ void __launch_bounds__(1024) offsets_scan_kernel(const int32_t* __restrict__ cnt, int n, int32_t* __restrict__ offset)
{
    __shared__ int wsum[32];
    __shared__ int carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += 1024) {
        const int i = i0 + threadIdx.x;
        const int v = i < n ? cnt[i] : 0;
        int s = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += u;
        }
        if (lane == 31) wsum[warp] = s;
        __syncthreads();
        if (warp == 0) {
            int w = wsum[lane];
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += u;
            }
            wsum[lane] = w;
        }
        __syncthreads();
        const int before = carry + (warp ? wsum[warp - 1] : 0) + s - v;
        if (i < n) offset[i] = before;
        __syncthreads();
        if (threadIdx.x == 1023) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) offset[n] = carry;
}

void launch_offsets_scan(const int32_t* cnt, int n, int32_t* offset, cudaStream_t st)
{
    offsets_scan_kernel<<<1, 1024, 0, st>>>(cnt, n, offset);
    count_launch();
}

// Second half of the fused path: block b of pair p copies its compacted (queryIdx, trainIdx, D1) rows from its slice of the
// scratch table to their final packed position and gathers the two keypoints of every match.
__global__ void __launch_bounds__(256) gather_packed_kernel(const int32_t* __restrict__ pairs, const float* __restrict__ xy, int feat_stride,
                                                            const int32_t* __restrict__ stage, const int32_t* __restrict__ blk_count, int bpp,
                                                            const int32_t* __restrict__ offset, int32_t* __restrict__ out_match,
                                                            float* __restrict__ out_corr)
{
    __shared__ int base_s;
    const int b = blockIdx.x, p = b / bpp, bi = b - p * bpp;
    const int n = blk_count[b];
    if (n == 0) return;
    if (threadIdx.x < 32) {
        int v = 0;
        for (int j = threadIdx.x; j < bi; j += 32) v += blk_count[p * bpp + j];
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) base_s = offset[p] + v;
    }
    __syncthreads();
    if ((int)threadIdx.x >= n) return;
    const int32_t* src = stage + (long long)b * 256 * 4 + 3 * threadIdx.x;
    const int q = src[0], t = src[1], d = src[2];
    const long long o = (long long)base_s + threadIdx.x;
    out_match[o * 3 + 0] = q;
    out_match[o * 3 + 1] = t;
    out_match[o * 3 + 2] = d;
    if (out_corr) {
        const int img_q = pairs[2 * p], img_t = pairs[2 * p + 1];
        const float2 a = reinterpret_cast<const float2*>(xy)[(long long)img_q * feat_stride + q];
        const float2 c = reinterpret_cast<const float2*>(xy)[(long long)img_t * feat_stride + t];
        reinterpret_cast<float4*>(out_corr)[o] = make_float4(a.x, a.y, c.x, c.y);
    }
}

int launch_match_tc(const sfm_bank* b, const int32_t* pairs, int n_pairs, int grid_req, int32_t* knn_out, int32_t* dbg_acc,
                    int dbg_mode, const Prefilter& pf, cudaStream_t st);
int launch_refine_filter(const sfm_bank* b, const int32_t* pairs, int n_pairs, int32_t* knn_out, const sfm_filter_params* prm,
                         const int32_t* knn_rev, int32_t* blk_count, int32_t* pair_count, cudaStream_t st);

}  // namespace sfm

using namespace sfm;

// The parameter checks every filter entry point shares.  `scratch` (the sweep records) and `out_corr` may be NULL; `packed`
// outputs address their rows with int32 offsets.
static int check_filter_args(const char* fn, const sfm_bank* bank, int n_pairs, const sfm_filter_params* prm, const int32_t* knn_rev,
                             const int32_t* scratch, const float* out_corr, bool packed)
{
    SFM_REQUIRE(n_pairs >= 0, "%s: negative pair count", fn);
    SFM_REQUIRE(!packed || (long long)n_pairs * bank->L.feat_stride < (1ll << 31), "%s: batch too large for int32 offsets", fn);
    SFM_REQUIRE(!prm->mutual || knn_rev, "%s: mutual check needs the reverse direction's kNN table", fn);
    SFM_REQUIRE(prm->ratio_mode >= SFM_RATIO_NONE && prm->ratio_mode <= SFM_RATIO_EXACT_INT, "%s: unknown ratio mode %d", fn, prm->ratio_mode);
    if (prm->ratio_mode == SFM_RATIO_EXACT_INT)
        SFM_REQUIRE(prm->ratio_num > 0 && prm->ratio_den > 0 && prm->ratio_num < 4096 && prm->ratio_den < 4096,
                    "%s: exact_int ratio needs 0 < num, den < 4096", fn);
    SFM_REQUIRE(((uintptr_t)scratch & 15) == 0, "%s: scratch must be 16-byte aligned", fn);
    SFM_REQUIRE(((uintptr_t)out_corr & 15) == 0, "%s: out_corr must be 16-byte aligned", fn);
    return SFM_OK;
}

// Refinement + filter -> offsets -> gather for n_pairs > 0, arguments checked, on the bank's device.
static int refine_filter_gather(const sfm_bank* bank, const int32_t* pairs_dev, int n_pairs, const sfm_filter_params* prm,
                                const int32_t* knn_rev, int32_t* scratch, int32_t* blk_count, int32_t* out_count, int32_t* out_offset,
                                int32_t* out_match, float* out_corr, cudaStream_t st)
{
    int rc = launch_refine_filter(bank, pairs_dev, n_pairs, scratch, prm, knn_rev, blk_count, out_count, st);
    if (rc) return rc;
    const int bpp = (int)(bank->L.feat_stride / 256);
    offsets_scan_kernel<<<1, 1024, 0, st>>>(out_count, n_pairs, out_offset);
    gather_packed_kernel<<<(unsigned)((long long)n_pairs * bpp), 256, 0, st>>>(pairs_dev, bank->xy, (int)bank->L.feat_stride, scratch, blk_count, bpp,
                                                                              out_offset, out_match, out_corr);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch(2);
    return SFM_OK;
}

// Sweep -> fused refinement + filter -> offsets -> gather: the matcher of the throughput path.  Output identical to
// sfm_match_knn2 + sfm_filter_matches_packed with the same parameters.
extern "C" int sfm_match_pairs_packed(const sfm_bank_t* bank, const int32_t* pairs_dev, int n_pairs, const sfm_match_params* mp,
                                      const sfm_filter_params* prm, const int32_t* knn_rev, int32_t* scratch, int32_t* blk_count,
                                      int32_t* out_count, int32_t* out_offset, int32_t* out_match, float* out_corr, void* stream)
{
    SFM_REQUIRE(bank && pairs_dev && prm && scratch && blk_count && out_count && out_offset && out_match, "sfm_match_pairs_packed: NULL argument");
    SFM_REQUIRE(bank->metric == SFM_METRIC_L2, "sfm_match_pairs_packed: bank metric is not L2");
    int rc = check_filter_args("sfm_match_pairs_packed", bank, n_pairs, prm, knn_rev, scratch, out_corr, true);
    if (rc) return rc;
    SFM_REQUIRE(!mp || mp->impl == SFM_MATCH_AUTO || mp->impl == SFM_MATCH_TCGEN05, "the fused path runs on the tcgen05 kernel");
    if (bank->n_filled <= 0) {
        set_error("sfm_match_pairs_packed: bank is empty");
        return SFM_ERR_STATE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SFM_ON_DEVICE(bank->device);
    if (n_pairs == 0) {
        SFM_CUDA_CHECK(cudaMemsetAsync(out_offset, 0, sizeof(int32_t), st));
        return SFM_OK;
    }
    Prefilter pf{SFM_RATIO_NONE, 1.0, 1, 1};
    if (mp && mp->prefilter_mode != SFM_RATIO_NONE) {
        // the sweep may only drop rows that fail THIS filter's ratio test
        SFM_REQUIRE(mp->prefilter_mode == prm->ratio_mode, "prefilter mode must equal the filter's ratio mode");
        pf.mode = mp->prefilter_mode;
        pf.ratio = mp->prefilter_ratio;
        pf.num2 = (long long)mp->prefilter_num * mp->prefilter_num;
        pf.den2 = (long long)mp->prefilter_den * mp->prefilter_den;
        if (pf.mode == SFM_RATIO_CV2_F32) SFM_REQUIRE(pf.ratio == prm->ratio, "prefilter ratio must equal the filter's ratio");
        else SFM_REQUIRE(pf.num2 * prm->ratio_den * prm->ratio_den == pf.den2 * prm->ratio_num * prm->ratio_num, "prefilter ratio must equal the filter's ratio");
    }
    rc = launch_match_tc(bank, pairs_dev, n_pairs, mp ? mp->grid : 0, scratch, nullptr, 3, pf, st);     // sweep only: records stay in scratch
    if (rc) return rc;
    return refine_filter_gather(bank, pairs_dev, n_pairs, prm, knn_rev, scratch, blk_count, out_count, out_offset, out_match, out_corr, st);
}

// The second half of sfm_match_pairs_packed on its own: `scratch` holds the candidate records of a sweep
// (sfm_match_knn2 with sweep_only = 4 and the same prefilter).  Lets a caller put the sweep of the NEXT batch on one stream and
// this batch's refinement / filter / gather on another (sfm_b200/plan.py).
extern "C" int sfm_refine_filter_packed(const sfm_bank_t* bank, const int32_t* pairs_dev, int n_pairs, const sfm_filter_params* prm,
                                        const int32_t* knn_rev, int32_t* scratch, int32_t* blk_count, int32_t* out_count, int32_t* out_offset,
                                        int32_t* out_match, float* out_corr, void* stream)
{
    SFM_REQUIRE(bank && pairs_dev && prm && scratch && blk_count && out_count && out_offset && out_match, "sfm_refine_filter_packed: NULL argument");
    SFM_REQUIRE(bank->metric == SFM_METRIC_L2, "sfm_refine_filter_packed: bank metric is not L2");
    int rc = check_filter_args("sfm_refine_filter_packed", bank, n_pairs, prm, knn_rev, scratch, out_corr, true);
    if (rc) return rc;
    if (bank->n_filled <= 0) {
        set_error("sfm_refine_filter_packed: bank is empty");
        return SFM_ERR_STATE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SFM_ON_DEVICE(bank->device);
    if (n_pairs == 0) {
        SFM_CUDA_CHECK(cudaMemsetAsync(out_offset, 0, sizeof(int32_t), st));
        return SFM_OK;
    }
    return refine_filter_gather(bank, pairs_dev, n_pairs, prm, knn_rev, scratch, blk_count, out_count, out_offset, out_match, out_corr, st);
}

extern "C" int sfm_filter_matches(const sfm_bank_t* bank, const int32_t* pairs_dev, int n_pairs, const int32_t* knn_fwd,
                                  const int32_t* knn_rev, const sfm_filter_params* prm, int32_t* out_count,
                                  int32_t* out_match, float* out_corr, void* stream)
{
    SFM_REQUIRE(bank && pairs_dev && knn_fwd && prm && out_count && out_match, "sfm_filter_matches: NULL argument");
    int rc = check_filter_args("sfm_filter_matches", bank, n_pairs, prm, knn_rev, nullptr, out_corr, false);
    if (rc) return rc;
    if (n_pairs == 0) return SFM_OK;
    SFM_ON_DEVICE(bank->device);
    filter_kernel<true><<<n_pairs, 256, 0, (cudaStream_t)stream>>>(
        pairs_dev, bank->count, bank->xy, (int)bank->L.feat_stride, knn_fwd, knn_rev, prm->ratio_mode, prm->mutual, prm->ratio,
        prm->ratio_num * prm->ratio_num, prm->ratio_den * prm->ratio_den, prm->max_distance_sq, out_count, nullptr, out_match,
        out_corr);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return SFM_OK;
}

// Packed layout: pair p's matches occupy rows [out_offset[p], out_offset[p+1]) of out_match / out_corr.
// Three launches: count, scan, write (the filter is ~1 % of the step; recomputing it beats a P x cap staging buffer).
extern "C" int sfm_filter_matches_packed(const sfm_bank_t* bank, const int32_t* pairs_dev, int n_pairs, const int32_t* knn_fwd,
                                         const int32_t* knn_rev, const sfm_filter_params* prm, int32_t* out_count,
                                         int32_t* out_offset, int32_t* out_match, float* out_corr, void* stream)
{
    SFM_REQUIRE(bank && pairs_dev && knn_fwd && prm && out_count && out_offset && out_match,
                "sfm_filter_matches_packed: NULL argument");
    int rc = check_filter_args("sfm_filter_matches_packed", bank, n_pairs, prm, knn_rev, nullptr, out_corr, true);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    SFM_ON_DEVICE(bank->device);
    if (n_pairs == 0) {
        SFM_CUDA_CHECK(cudaMemsetAsync(out_offset, 0, sizeof(int32_t), st));
        return SFM_OK;
    }
    const long long num2 = prm->ratio_num * prm->ratio_num, den2 = prm->ratio_den * prm->ratio_den;
    filter_kernel<false><<<n_pairs, 256, 0, st>>>(pairs_dev, bank->count, bank->xy, (int)bank->L.feat_stride, knn_fwd, knn_rev,
                                                  prm->ratio_mode, prm->mutual, prm->ratio, num2, den2, prm->max_distance_sq,
                                                  out_count, nullptr, nullptr, nullptr);
    offsets_scan_kernel<<<1, 1024, 0, st>>>(out_count, n_pairs, out_offset);
    filter_kernel<true><<<n_pairs, 256, 0, st>>>(pairs_dev, bank->count, bank->xy, (int)bank->L.feat_stride, knn_fwd, knn_rev,
                                                 prm->ratio_mode, prm->mutual, prm->ratio, num2, den2, prm->max_distance_sq,
                                                 nullptr, out_offset, out_match, out_corr);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch(3);
    return SFM_OK;
}
