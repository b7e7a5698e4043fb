// ransac_h.cu -- batched RANSAC homography estimation (SURVEY.md §8f rank 2).  Compile with -fmad=false.
//
// Second model of the geometric-verification stage the reference left empty (code/geometric_verification.py is a
// 0-byte file; placeholder at code/pipeline.py:60-65): planar / panoramic pairs are explained by a homography, and the
// H-vs-F inlier ratio classifies the pair for the scene graph.  Conventions follow cv2.findHomography(RANSAC):
// x2 ~ H x1, H[8] normalised to 1, uint8 inlier mask, inlier iff |proj(H x1) - x2|^2 <= thr^2.
//
// The kernel body is ransac_driver (ransac_common.cuh), shared with RANSAC-F.  This file supplies the homography model:
//   solve   A: 4-point sample, lane r holds row r of the 8 x 9 DLT system (point r / 2, x- or y-equation), one null vector
//           B: denormalise; the sample points must keep the sign of the projective depth (needs the sample again)
//   score   forward transfer error
//   stop    the caller's optional stop target (stop_target)
//   LO      normalised DLT on the inliers, two rows per inlier
// Bit-identical to oracle/ransac_h.c.
#include "ransac_common.cuh"

namespace sfm {

// H = T2^-1 Hn T1 with T = [s 0 -s*cx; 0 s -s*cy; 0 0 1], scaled to unit Frobenius norm
static __device__ int denormalise_h(const double* Hn, Norm2d n1, Norm2d n2, double* H)
{
    double G[9];
    for (int r = 0; r < 3; ++r) {
        const double h0 = Hn[r * 3 + 0], h1 = Hn[r * 3 + 1], h2 = Hn[r * 3 + 2];
        G[r * 3 + 0] = n1.s * h0;
        G[r * 3 + 1] = n1.s * h1;
        G[r * 3 + 2] = h2 - n1.s * (n1.cx * h0 + n1.cy * h1);
    }
    const double is2 = 1.0 / n2.s;
    for (int c = 0; c < 3; ++c) {
        const double g0 = G[0 + c], g1 = G[3 + c], g2 = G[6 + c];
        H[0 + c] = is2 * g0 + n2.cx * g2;
        H[3 + c] = is2 * g1 + n2.cy * g2;
        H[6 + c] = g2;
    }
    double ss = 0.0;
    for (int i = 0; i < 9; ++i) ss += H[i] * H[i];
    if (!(ss > 0.0) || !(ss < 1e300)) return 0;
    const double inv = 1.0 / sqrt(ss);
    for (int i = 0; i < 9; ++i) H[i] *= inv;
    return 1;
}

// Minimal solver, phase A (8 lanes per hypothesis): Hartley normalisation of the 4 sample points (every lane computes
// the same values), lane r builds row r of the 8 x 9 DLT system (point r / 2, x- or y-equation), the octet eliminates
// it cooperatively; out[0..8] = null vector (normalised frame), out[18..23] = n1, n2.
static __device__ __forceinline__ bool solve_h_null_space(const Pts& pts, const int* idx, int sl, unsigned gmask, double* out)
{
    Norm2d n1, n2;
    double u1, v1, u2, v2;                    // (the 0.25 of the 4-point mean is 1.0 / 4, bit for bit)
    if (!hartley_sample<4>(pts, idx, sl >> 1, n1, n2, u1, v1, u2, v2)) return false;
    double a[9];
    if (sl & 1) {
        a[0] = 0.0; a[1] = 0.0; a[2] = 0.0; a[3] = u1; a[4] = v1; a[5] = 1.0;
        a[6] = -(v2 * u1); a[7] = -(v2 * v1); a[8] = -v2;
    } else {
        a[0] = u1; a[1] = v1; a[2] = 1.0; a[3] = 0.0; a[4] = 0.0; a[5] = 0.0;
        a[6] = -(u2 * u1); a[7] = -(u2 * v1); a[8] = -u2;
    }
    CoopGJ st;
    if (!coop_gauss_jordan<8>(a, sl, gmask, 1e-10, st)) return false;
    coop_null_vector<8>(a, sl, st, 0, out);
    if (sl == 0) store_norms(out, n1, n2);
    return true;
}

// Minimal solver, phase B (one thread per hypothesis): denormalise, then the four sample points must lie on one side
// of the line H maps to infinity (orientation is preserved)
static __device__ int model_from_null_space_h(const double* in, const Pts& pts, const int* idx, double* Hout)
{
    double Hn[9];
    for (int i = 0; i < 9; ++i) Hn[i] = in[i];
    Norm2d n1, n2;
    load_norms(in, n1, n2);
    if (!denormalise_h(Hn, n1, n2, Hout)) return 0;
    int pos = 0, neg = 0;
    for (int k = 0; k < 4; ++k) {
        const float4 c = pts[idx[k]];
        const double w = Hout[6] * (double)c.x + Hout[7] * (double)c.y + Hout[8];
        pos += (w > 0.0);
        neg += (w < 0.0);
    }
    return (pos == 4 || neg == 4) ? 1 : 0;
}

// fp32, division-free forward transfer error: |H x1 - w x2|^2 <= thr^2 w^2
static __device__ __forceinline__ bool is_inlier_h(const float (&H)[9], const float4 c, float thr2)
{
    const float X = fmaf(H[0], c.x, fmaf(H[1], c.y, H[2]));
    const float Y = fmaf(H[3], c.x, fmaf(H[4], c.y, H[5]));
    const float W = fmaf(H[6], c.x, fmaf(H[7], c.y, H[8]));
    const float ex = fmaf(-c.z, W, X);
    const float ey = fmaf(-c.w, W, Y);
    const float ey2 = ey * ey;
    const float e2 = fmaf(ex, ex, ey2);
    const float lim = thr2 * (W * W);
    return e2 <= lim && lim > 0.f;
}

struct HomographyModel {
    static constexpr const char* kName = "sfm_ransac_h";
    static constexpr int kMaxSample = 4, kRoots = 1, kLoMin = 4;
    static constexpr bool kSampleInPhaseB = true;                          // the orientation check reads the sample points

    static int check(const sfm_ransac_params&) { return SFM_OK; }          // solver and score are not used
    static __device__ __forceinline__ int sample_size(const sfm_ransac_params&) { return 4; }
    static __device__ __forceinline__ bool null_space(const Pts& pts, const int* idx, int, int sl, unsigned gmask, double* out)
    {
        return solve_h_null_space(pts, idx, sl, gmask, out);
    }
    static __device__ __forceinline__ int models(const double* in, int, const Pts& pts, const int* idx, double* out)
    {
        return model_from_null_space_h(in, pts, idx, out);
    }
    static __device__ __forceinline__ bool inlier(const float (&H)[9], const float4 c, float thr2, int)
    {
        return is_inlier_h(H, c, thr2);
    }
    // the two DLT rows of each inlier
    static __device__ __forceinline__ void lo_rows(double (&acc)[45], double u1, double v1, double u2, double v2)
    {
        const double ra[9] = {u1, v1, 1.0, 0.0, 0.0, 0.0, -(u2 * u1), -(u2 * v1), -u2};
        const double rb[9] = {0.0, 0.0, 0.0, u1, v1, 1.0, -(v2 * u1), -(v2 * v1), -v2};
        int e = 0;
#pragma unroll
        for (int a = 0; a < 9; ++a)
#pragma unroll
            for (int b = a; b < 9; ++b) {
                acc[e] += ra[a] * ra[b];
                acc[e] += rb[a] * rb[b];
                ++e;
            }
    }
    static __device__ __forceinline__ int refit(double* Hn, Norm2d n1, Norm2d n2, double* H) { return denormalise_h(Hn, n1, n2, H); }
};

__global__ void __launch_bounds__(kRansacThreads, 2) ransac_h_kernel(
    const float* __restrict__ corr, int corr_stride, const int32_t* __restrict__ count, const int32_t* __restrict__ offsets,
    const uint32_t* __restrict__ pair_id, const uint32_t* __restrict__ samples, const int32_t* __restrict__ stop_target,
    sfm_ransac_params prm, int pts_cap, double* __restrict__ out_H, int32_t* __restrict__ out_ninl, uint8_t* __restrict__ out_mask,
    int32_t* __restrict__ out_iters)
{
    ransac_driver<HomographyModel>(corr, corr_stride, count, offsets, pair_id, samples, stop_target, prm, pts_cap, out_H, out_ninl,
                                   out_mask, out_iters);
}

}  // namespace sfm

using namespace sfm;

extern "C" int sfm_ransac_h_batch(const float* corr, int corr_stride, const int32_t* count, int n_pairs, const uint32_t* pair_id,
                                  const uint32_t* samples, const int32_t* stop_target, const sfm_ransac_params* prm, double* out_H,
                                  int32_t* out_ninl, uint8_t* out_mask, int32_t* out_iters, void* stream)
{
    SFM_REQUIRE(count != nullptr, "sfm_ransac_h_batch: NULL argument");
    return launch_ransac<HomographyModel>(ransac_h_kernel, corr, corr_stride, count, nullptr, n_pairs, pair_id, samples, stop_target, prm,
                                          out_H, out_ninl, out_mask, out_iters, stream);
}

extern "C" int sfm_ransac_h_packed(const float* corr, const int32_t* offsets, int n_pairs, int max_count, const uint32_t* pair_id,
                                   const uint32_t* samples, const int32_t* stop_target, const sfm_ransac_params* prm, double* out_H,
                                   int32_t* out_ninl, uint8_t* out_mask, int32_t* out_iters, void* stream)
{
    SFM_REQUIRE(offsets != nullptr, "sfm_ransac_h_packed: NULL argument");
    return launch_ransac<HomographyModel>(ransac_h_kernel, corr, max_count, nullptr, offsets, n_pairs, pair_id, samples, stop_target, prm,
                                          out_H, out_ninl, out_mask, out_iters, stream);
}
