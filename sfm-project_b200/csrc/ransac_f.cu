// ransac_f.cu -- batched RANSAC fundamental-matrix verification (K4).  Compile with -fmad=false.
//
// Fills the reference's empty code/geometric_verification.py (0 bytes; placeholder at
// code/pipeline.py:60) with the conventions of cv2.findFundamentalMat(FM_RANSAC): x2^T F x1 = 0,
// F[8] normalised to 1, uint8 inlier mask, inlier iff max(d1^2, d2^2) <= thr^2 (SURVEY.md A.4).
//
// The kernel body is ransac_driver (ransac_common.cuh).  This file supplies the fundamental-matrix model:
//   solve   A: one epipolar row per lane, 9 - m null vectors (m = 7 or 8 sample points)
//           B: rank-2 projection (8-point) or cubic in the pencil (7-point, <= 3 models)
//   score   symmetric epipolar distance (cv2) or Sampson
//   LO      normalised 8-point refit on the inliers, rank 2 enforced
// Every floating-point operation is IEEE basic arithmetic in a fixed order (explicit fma only), so masks and counts are
// bit-identical to oracle/ransac_f.c, which tests/ use as the checker.
#include <math.h>

#include "ransac_common.cuh"

namespace sfm {

__device__ double det3(const double* r0, const double* r1, const double* r2)
{
    const double a = r1[1] * r2[2] - r1[2] * r2[1];
    const double b = r1[0] * r2[2] - r1[2] * r2[0];
    const double c = r1[0] * r2[1] - r1[1] * r2[0];
    return r0[0] * a - r0[1] * b + r0[2] * c;
}

__device__ void enforce_rank2(double* F)
{
    double G[9], V[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) G[i * 3 + j] = F[0 + i] * F[0 + j] + F[3 + i] * F[3 + j] + F[6 + i] * F[6 + j];
    jacobi_eig_n<3>(G, V, 6);
    // smallest eigenvalue -> its eigenvector (column k of V), selected without dynamic indexing
    int k = 0;
    if (G[4] < G[0]) k = 1;
    if (G[8] < (k ? G[4] : G[0])) k = 2;
    const double v0 = k == 0 ? V[0] : (k == 1 ? V[1] : V[2]);
    const double v1 = k == 0 ? V[3] : (k == 1 ? V[4] : V[5]);
    const double v2 = k == 0 ? V[6] : (k == 1 ? V[7] : V[8]);
    for (int r = 0; r < 3; ++r) {
        const double w = F[r * 3 + 0] * v0 + F[r * 3 + 1] * v1 + F[r * 3 + 2] * v2;
        F[r * 3 + 0] -= w * v0;
        F[r * 3 + 1] -= w * v1;
        F[r * 3 + 2] -= w * v2;
    }
}

__device__ int denormalise(const double* Fh, Norm2d n1, Norm2d n2, double* F)
{
    double G[9];
    for (int r = 0; r < 3; ++r) {
        const double f0 = Fh[r * 3 + 0], f1 = Fh[r * 3 + 1], f2 = Fh[r * 3 + 2];
        G[r * 3 + 0] = n1.s * f0;
        G[r * 3 + 1] = n1.s * f1;
        G[r * 3 + 2] = f2 - n1.s * (n1.cx * f0 + n1.cy * f1);
    }
    for (int c = 0; c < 3; ++c) {
        const double g0 = G[0 + c], g1 = G[3 + c], g2 = G[6 + c];
        F[0 + c] = n2.s * g0;
        F[3 + c] = n2.s * g1;
        F[6 + c] = g2 - n2.s * (n2.cx * g0 + n2.cy * g1);
    }
    double ss = 0.0;
    for (int i = 0; i < 9; ++i) ss += F[i] * F[i];
    if (!(ss > 0.0) || !(ss < 1e300)) return 0;
    const double inv = 1.0 / sqrt(ss);
    for (int i = 0; i < 9; ++i) F[i] *= inv;
    return 1;
}

__device__ int solve_cubic(double c3, double c2, double c1, double c0, double* roots)
{
    const double mx = fmax(fabs(c2), fmax(fabs(c1), fabs(c0)));
    int n = 0;
    if (!(fabs(c3) > 1e-14 * mx)) {
        if (!(fabs(c2) > 1e-14 * fmax(fabs(c1), fabs(c0)))) {
            if (c1 != 0.0) roots[n++] = -c0 / c1;
            return n;
        }
        const double disc = c1 * c1 - 4.0 * c2 * c0;
        if (disc < 0.0) return 0;
        const double sq = sqrt(disc);
        const double q = -0.5 * (c1 + (c1 >= 0.0 ? sq : -sq));
        roots[n++] = q / c2;
        if (q != 0.0) roots[n++] = c0 / q;
        return n;
    }
    const double b = c2 / c3, c = c1 / c3, d = c0 / c3;
    const double R = 1.0 + fmax(fabs(b), fmax(fabs(c), fabs(d)));
    double lo = -R, hi = R;
    for (int it = 0; it < 80; ++it) {
        const double mid = 0.5 * (lo + hi);
        const double fm = ((mid + b) * mid + c) * mid + d;
        if (fm < 0.0) lo = mid; else hi = mid;
    }
    double r = 0.5 * (lo + hi);
    for (int it = 0; it < 2; ++it) {
        const double f = ((r + b) * r + c) * r + d;
        const double fp = (3.0 * r + 2.0 * b) * r + c;
        if (fp != 0.0) r = r - f / fp;
    }
    roots[n++] = r;
    const double B = b + r;
    const double C = c + r * B;
    const double disc = B * B - 4.0 * C;
    if (disc >= 0.0) {
        const double sq = sqrt(disc);
        const double q = -0.5 * (B + (B >= 0.0 ? sq : -sq));
        double r2 = q;
        double r3 = (q != 0.0) ? C / q : q;
        for (int it = 0; it < 2; ++it) {
            double f = ((r2 + b) * r2 + c) * r2 + d;
            double fp = (3.0 * r2 + 2.0 * b) * r2 + c;
            if (fp != 0.0) r2 = r2 - f / fp;
            f = ((r3 + b) * r3 + c) * r3 + d;
            fp = (3.0 * r3 + 2.0 * b) * r3 + c;
            if (fp != 0.0) r3 = r3 - f / fp;
        }
        roots[n++] = r2;
        roots[n++] = r3;
    }
    return n;
}

// Minimal solver, phase A (8 lanes per hypothesis): Hartley normalisation of the m sample points (every lane computes
// the same values), lane r builds row r of the m x 9 epipolar system, the octet eliminates it cooperatively and the
// null space (9 - m vectors) plus the two normalisations land in shared memory: out[0..17] = N, out[18..23] = n1, n2.
template <int M>
static __device__ __forceinline__ bool solve_null_space(const Pts& pts, const int* idx, int sl, unsigned gmask, double* out)
{
    Norm2d n1, n2;
    double u1, v1, u2, v2;                                                 // this lane's sample point
    if (!hartley_sample<M>(pts, idx, sl, n1, n2, u1, v1, u2, v2)) return false;
    double a[9] = {u2 * u1, u2 * v1, u2, v2 * u1, v2 * v1, v2, u1, v1, 1.0};
    CoopGJ st;
    if (!coop_gauss_jordan<M>(a, sl, gmask, 1e-12, st)) return false;
#pragma unroll
    for (int c = 0; c < 9 - M; ++c) coop_null_vector<M>(a, sl, st, c, out + 9 * c);
    if (sl == 0) store_norms(out, n1, n2);
    return true;
}

// Minimal solver, phase B (one thread per hypothesis): null space -> up to 3 unit-Frobenius-norm F
static __device__ int models_from_null_space(const double* in, int m, double* Fout)
{
    double N[2][9];
    for (int i = 0; i < 9; ++i) { N[0][i] = in[i]; N[1][i] = in[9 + i]; }
    Norm2d n1, n2;
    load_norms(in, n1, n2);
    if (m == 8) {
        double Fh[9];
        for (int i = 0; i < 9; ++i) Fh[i] = N[0][i];
        enforce_rank2(Fh);
        return denormalise(Fh, n1, n2, Fout);
    }
    const double* F1 = N[0];
    const double* F2 = N[1];
    const double c3 = det3(F1, F1 + 3, F1 + 6);
    const double c0 = det3(F2, F2 + 3, F2 + 6);
    const double c2 = det3(F2, F1 + 3, F1 + 6) + det3(F1, F2 + 3, F1 + 6) + det3(F1, F1 + 3, F2 + 6);
    const double c1 = det3(F1, F2 + 3, F2 + 6) + det3(F2, F1 + 3, F2 + 6) + det3(F2, F2 + 3, F1 + 6);
    double roots[3];
    const int nr = solve_cubic(c3, c2, c1, c0, roots);
    int nm = 0;
    for (int r = 0; r < nr; ++r) {
        double Fh[9];
        for (int i = 0; i < 9; ++i) Fh[i] = roots[r] * F1[i] + F2[i];
        if (denormalise(Fh, n1, n2, Fout + 9 * nm)) ++nm;
    }
    return nm;
}

// fp32, division-free: num^2 <= thr^2 * min(|l2|^2, |l1|^2)  (cv2 metric)  or  thr^2 * (|l2|^2 + |l1|^2)  (Sampson)
__device__ __forceinline__ bool is_inlier(const float (&F)[9], const float4 c, float thr2, int score)
{
    const float a = fmaf(F[0], c.x, fmaf(F[1], c.y, F[2]));
    const float b = fmaf(F[3], c.x, fmaf(F[4], c.y, F[5]));
    const float cc = fmaf(F[6], c.x, fmaf(F[7], c.y, F[8]));
    const float num = fmaf(c.z, a, fmaf(c.w, b, cc));
    const float a2 = fmaf(F[0], c.z, fmaf(F[3], c.w, F[6]));
    const float b2 = fmaf(F[1], c.z, fmaf(F[4], c.w, F[7]));
    const float bb = b * b;
    const float s1 = fmaf(a, a, bb);
    const float bb2 = b2 * b2;
    const float s2 = fmaf(a2, a2, bb2);
    const float n2 = num * num;
    const float lim = (score == SFM_SCORE_SAMPSON) ? thr2 * (s1 + s2) : thr2 * fminf(s1, s2);
    return n2 <= lim;
}

struct FundamentalModel {
    static constexpr const char* kName = "sfm_ransac_f";
    static constexpr int kMaxSample = 8, kRoots = 3, kLoMin = 8;           // LO needs 8 inliers for the 7-point solver too
    static constexpr bool kSampleInPhaseB = false;

    static int check(const sfm_ransac_params& prm)
    {
        SFM_REQUIRE(prm.solver == SFM_SOLVER_7PT || prm.solver == SFM_SOLVER_8PT, "solver must be 7 or 8, got %d", prm.solver);
        SFM_REQUIRE(prm.score == SFM_SCORE_SYM_EPIPOLAR || prm.score == SFM_SCORE_SAMPSON, "unknown score %d", prm.score);
        return SFM_OK;
    }
    static __device__ __forceinline__ int sample_size(const sfm_ransac_params& prm) { return prm.solver; }
    static __device__ __forceinline__ bool null_space(const Pts& pts, const int* idx, int m, int sl, unsigned gmask, double* out)
    {
        return (m == 8) ? solve_null_space<8>(pts, idx, sl, gmask, out) : solve_null_space<7>(pts, idx, sl, gmask, out);
    }
    static __device__ __forceinline__ int models(const double* in, int m, const Pts&, const int*, double* out)
    {
        return models_from_null_space(in, m, out);
    }
    static __device__ __forceinline__ bool inlier(const float (&F)[9], const float4 c, float thr2, int score)
    {
        return is_inlier(F, c, thr2, score);
    }
    // one epipolar row r per inlier: r (x) r
    static __device__ __forceinline__ void lo_rows(double (&acc)[45], double u1, double v1, double u2, double v2)
    {
        const double r[9] = {u2 * u1, u2 * v1, u2, v2 * u1, v2 * v1, v2, u1, v1, 1.0};
        int e = 0;
#pragma unroll
        for (int a = 0; a < 9; ++a)
#pragma unroll
            for (int b = a; b < 9; ++b) acc[e++] += r[a] * r[b];
    }
    static __device__ __forceinline__ int refit(double* Fh, Norm2d n1, Norm2d n2, double* F)
    {
        enforce_rank2(Fh);
        return denormalise(Fh, n1, n2, F);
    }
};

__global__ void __launch_bounds__(kRansacThreads, 2) ransac_f_kernel(
    const float* __restrict__ corr, int corr_stride, const int32_t* __restrict__ count, const int32_t* __restrict__ offsets,
    const uint32_t* __restrict__ pair_id, const uint32_t* __restrict__ samples, const int32_t* __restrict__ /* stop_target */,
    sfm_ransac_params prm, int pts_cap, double* __restrict__ out_F, int32_t* __restrict__ out_ninl, uint8_t* __restrict__ out_mask,
    int32_t* __restrict__ out_iters)
{
    ransac_driver<FundamentalModel>(corr, corr_stride, count, offsets, pair_id, samples, nullptr, prm, pts_cap, out_F, out_ninl,
                                    out_mask, out_iters);
}

}  // namespace sfm

using namespace sfm;

extern "C" int sfm_ransac_f_batch(const float* corr, int corr_stride, const int32_t* count, int n_pairs, const uint32_t* pair_id,
                                  const uint32_t* samples, const sfm_ransac_params* prm, double* out_F, int32_t* out_ninl,
                                  uint8_t* out_mask, int32_t* out_iters, void* stream)
{
    SFM_REQUIRE(count != nullptr, "sfm_ransac_f_batch: NULL argument");
    return launch_ransac<FundamentalModel>(ransac_f_kernel, corr, corr_stride, count, nullptr, n_pairs, pair_id, samples, nullptr, prm,
                                           out_F, out_ninl, out_mask, out_iters, stream);
}

extern "C" int sfm_ransac_f_packed(const float* corr, const int32_t* offsets, int n_pairs, int max_count, const uint32_t* pair_id,
                                   const uint32_t* samples, const sfm_ransac_params* prm, double* out_F, int32_t* out_ninl,
                                   uint8_t* out_mask, int32_t* out_iters, void* stream)
{
    SFM_REQUIRE(offsets != nullptr, "sfm_ransac_f_packed: NULL argument");
    return launch_ransac<FundamentalModel>(ransac_f_kernel, corr, max_count, nullptr, offsets, n_pairs, pair_id, samples, nullptr, prm,
                                           out_F, out_ninl, out_mask, out_iters, stream);
}
