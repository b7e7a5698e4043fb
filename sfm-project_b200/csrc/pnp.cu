// pnp.cu -- registration: camera poses from 2-D / 3-D correspondences (batched RANSAC-PnP).  Compile with -fmad=false.
//
// include/sfm_b200.h, "absolute pose / registration", states the contract.  Two kernels:
//   pnp_gather_kernel   one CTA per query: the features of the query's image whose track has a point, compacted in feature
//                       order (ballot ranks within a warp, warp totals in warp order) into the strided correspondence layout
//   pnp_ransac_kernel   one 256-thread CTA per query, shaped like ransac_driver (ransac_common.cuh):
//     stage    the first kPnpCap correspondences as (x^, y^) and X in shared memory; a wider query reads the tail via L1/L2
//     solve    one thread per hypothesis: Lambda Twist P3P, up to 4 poses into shared memory
//     score    one warp per pair of poses, lanes stride over the correspondences, counts reduced by shuffles
//     select   strict-greater argmax in (hypothesis, root) order, then the adaptive stop rule
//     refine   Gauss-Newton on the pixel residuals of the inliers: 28 sums per step through block_tree_sum_many, the 6 x 6
//              solve repeated by every thread on the same totals (no broadcast)
// fp64 throughout, IEEE basic operations and sqrt in a fixed order: bit-identical to oracle/pnp.c.
#include <algorithm>

#include "ransac_common.cuh"

namespace sfm {

constexpr int kPnpCap = 4096;           // correspondences per query staged in shared memory
constexpr int kPnpRoots = 4;            // P3P poses per hypothesis
constexpr int kPnpGroup = 2;            // poses scored together by one warp
constexpr int kPnpSums = 28;            // Gauss-Newton sums: 21 of J^T J, 6 of J^T r, the cost

enum PnpStatus { kPnpOk = 0, kPnpFew = 1, kPnpNoModel = 2, kPnpFewInliers = 3, kPnpInvalid = 4, kPnpStatuses = 5 };

// ------------------------------------------------------------------------------------------------------------ gather
__global__ void __launch_bounds__(256) pnp_gather_kernel(int n_images, int S, const int32_t* __restrict__ track_of,
                                                         const int64_t* __restrict__ track_counts, long long max_tracks,
                                                         const uint8_t* __restrict__ point_status, const double* __restrict__ X,
                                                         const float* __restrict__ xy, int xy_stride, const int32_t* __restrict__ image,
                                                         float* __restrict__ out_xy, double* __restrict__ out_X,
                                                         int32_t* __restrict__ out_feature, int32_t* __restrict__ out_count)
{
    __shared__ int warp_total[8];
    const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int img = __ldg(image + q);
    if (img < 0 || img >= n_images) {
        if (tid == 0) out_count[q] = 0;
        return;
    }
    const long long n_tracks = min((long long)__ldg(track_counts), max_tracks);
    const long long o = (long long)q * S;
    int base = 0;
    for (int f0 = 0; f0 < S; f0 += 256) {
        const int f = f0 + tid;
        int k = -1;
        if (f < S) k = __ldg(track_of + (long long)img * S + f);
        const bool use = k >= 0 && k < n_tracks && __ldg(point_status + k) == 0;
        const unsigned bal = __ballot_sync(0xffffffffu, use);
        if (lane == 0) warp_total[warp] = __popc(bal);
        __syncthreads();
        int off = base, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const int c = warp_total[w];
            off += w < warp ? c : 0;
            total += c;
        }
        if (use) {
            const long long r = o + off + __popc(bal & ((1u << lane) - 1u));
            const float2 p = __ldg(reinterpret_cast<const float2*>(xy) + (long long)img * xy_stride + f);
            reinterpret_cast<float2*>(out_xy)[r] = p;
            out_X[3 * r + 0] = __ldg(X + 3ll * k + 0);
            out_X[3 * r + 1] = __ldg(X + 3ll * k + 1);
            out_X[3 * r + 2] = __ldg(X + 3ll * k + 2);
            out_feature[r] = f;
        }
        base += total;
        __syncthreads();                    // warp_total is rewritten by the next chunk
    }
    if (tid == 0) out_count[q] = base;
}

// ------------------------------------------------------------------------------------------------------------ P3P
static __device__ __forceinline__ bool is_finite(double v) { return fabs(v) <= 1.7976931348623157e308; }

// One real root of g^3 + b g^2 + c g + d (Lambda Twist's cubick): a start on the monotone side of a stationary point, then
// Newton steps (at least 7, at most 50, until |f| <= 1e-13).
static __device__ double p3p_cubic(double b, double c, double d)
{
    double r0;
    if (b * b >= 3.0 * c) {
        const double v = sqrt(b * b - 3.0 * c);
        const double t1 = (-b - v) / 3.0;
        double k = ((t1 + b) * t1 + c) * t1 + d;
        if (k > 0.0) {
            r0 = t1 - sqrt(-k / (3.0 * t1 + b));
        } else {
            const double t2 = (-b + v) / 3.0;
            k = ((t2 + b) * t2 + c) * t2 + d;
            r0 = t2 + sqrt(-k / (3.0 * t2 + b));
        }
    } else {
        r0 = -b / 3.0;
        if (fabs((3.0 * r0 + 2.0 * b) * r0 + c) < 1e-4) r0 = r0 + 1.0;
    }
#pragma unroll 1
    for (int it = 0; it < 50; ++it) {
        const double fx = ((r0 + b) * r0 + c) * r0 + d;
        if (!(it < 7 || fabs(fx) > 1e-13)) break;
        const double fpx = (3.0 * r0 + 2.0 * b) * r0 + c;
        r0 = r0 - fx / fpx;
    }
    return r0;
}

// At most 5 Gauss-Newton steps on the three depth equations; a step is kept only if |r|_1 does not grow.
static __device__ __forceinline__ void p3p_refine_depths(double (&L)[3], double a12, double a13, double a23, double b12, double b13,
                                                         double b23)
{
#pragma unroll 1
    for (int it = 0; it < 5; ++it) {
        const double l1 = L[0], l2 = L[1], l3 = L[2];
        const double r1 = l1 * l1 + l2 * l2 + b12 * l1 * l2 - a12;
        const double r2 = l1 * l1 + l3 * l3 + b13 * l1 * l3 - a13;
        const double r3 = l2 * l2 + l3 * l3 + b23 * l2 * l3 - a23;
        const double rs = fabs(r1) + fabs(r2) + fabs(r3);
        if (rs < 1e-10) break;
        const double v0 = 2.0 * l1 + b12 * l2, v1 = 2.0 * l2 + b12 * l1;
        const double v3 = 2.0 * l1 + b13 * l3, v5 = 2.0 * l3 + b13 * l1;
        const double v7 = 2.0 * l2 + b23 * l3, v8 = 2.0 * l3 + b23 * l2;
        const double det = 1.0 / (-v0 * v5 * v7 - v1 * v3 * v8);
        const double n1 = l1 - det * (-v5 * v7 * r1 + -v1 * v8 * r2 + v1 * v5 * r3);
        const double n2 = l2 - det * (-v3 * v8 * r1 + v0 * v8 * r2 + -v0 * v5 * r3);
        const double n3 = l3 - det * (v3 * v7 * r1 + -v0 * v7 * r2 + -v1 * v3 * r3);
        const double s1 = n1 * n1 + n2 * n2 + b12 * n1 * n2 - a12;
        const double s2 = n1 * n1 + n3 * n3 + b13 * n1 * n3 - a13;
        const double s3 = n2 * n2 + n3 * n3 + b23 * n2 * n3 - a23;
        if (fabs(s1) + fabs(s2) + fabs(s3) > rs) break;
        L[0] = n1; L[1] = n2; L[2] = n3;
    }
}

// Depths of the two lines of the degenerate conic for one sign s of the eigenvector combination; appends to Ls.
static __device__ __forceinline__ void p3p_line(double s, const double (&V)[9], int e0, int e1, double a12, double a13, double a23,
                                                double b12, double b13, double b23, double (&Ls)[4][3], int& n)
{
    const double w2 = 1.0 / (s * V[e1] - V[e0]);
    const double w0 = (V[3 + e0] - s * V[3 + e1]) * w2;
    const double w1 = (V[6 + e0] - s * V[6 + e1]) * w2;
    const double a = 1.0 / ((a13 - a12) * w1 * w1 - a12 * b13 * w1 - a12);
    const double b = (a13 * b12 * w1 - a12 * b13 * w0 - 2.0 * w0 * w1 * (a12 - a13)) * a;
    const double c = ((a13 - a12) * w0 * w0 + a13 * b12 * w0 + a13) * a;
    const double disc = b * b - 4.0 * c;
    if (!(disc >= 0.0)) return;
    const double y = sqrt(disc);
    const double tau1 = b < 0.0 ? 0.5 * (-b + y) : 0.5 * (-b - y);
    const double tau2 = c / tau1;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const double tau = k == 0 ? tau1 : tau2;
        if (!(tau > 0.0)) continue;
        const double d = a23 / (tau * (b23 + tau) + 1.0);
        if (!(d > 0.0)) continue;
        const double l2 = sqrt(d);
        const double l3 = tau * l2;
        const double l1 = w0 * l2 + w1 * l3;
        if (!(l1 >= 0.0)) continue;
        const int slot = n;             // at most 4 in total: two signs x two roots
        Ls[slot & 3][0] = l1; Ls[slot & 3][1] = l2; Ls[slot & 3][2] = l3;
        n = n + 1;
    }
}

// Lambda Twist P3P on three normalised observations (nx, ny) and world points X (row k = point k).  Writes up to 4 poses
// (12 doubles: R row-major, t) to out and returns their number.
static __device__ __noinline__ int p3p(const double (&nx)[3], const double (&ny)[3], const double (&X)[3][3], double* out)
{
    double y[3][3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double inv = 1.0 / sqrt(nx[k] * nx[k] + ny[k] * ny[k] + 1.0);
        y[k][0] = nx[k] * inv; y[k][1] = ny[k] * inv; y[k][2] = inv;
    }
    const double b12 = -2.0 * (y[0][0] * y[1][0] + y[0][1] * y[1][1] + y[0][2] * y[1][2]);
    const double b13 = -2.0 * (y[0][0] * y[2][0] + y[0][1] * y[2][1] + y[0][2] * y[2][2]);
    const double b23 = -2.0 * (y[1][0] * y[2][0] + y[1][1] * y[2][1] + y[1][2] * y[2][2]);
    double d12[3], d13[3], d23[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        d12[c] = X[0][c] - X[1][c];
        d13[c] = X[0][c] - X[2][c];
        d23[c] = X[1][c] - X[2][c];
    }
    const double a12 = d12[0] * d12[0] + d12[1] * d12[1] + d12[2] * d12[2];
    const double a13 = d13[0] * d13[0] + d13[1] * d13[1] + d13[2] * d13[2];
    const double a23 = d23[0] * d23[0] + d23[1] * d23[1] + d23[2] * d23[2];
    const double c31 = -0.5 * b13, c23 = -0.5 * b23, c12 = -0.5 * b12;
    const double blob = c12 * c23 * c31 - 1.0;
    const double s31 = 1.0 - c31 * c31, s23 = 1.0 - c23 * c23, s12 = 1.0 - c12 * c12;
    double p3 = a13 * (a23 * s31 - a13 * s23);
    double p2 = 2.0 * blob * a23 * a13 + a13 * (2.0 * a12 + a13) * s23 + a23 * (a23 - a12) * s31;
    double p1 = a23 * (a13 - a23) * s12 - a12 * a12 * s23 - 2.0 * a12 * (blob * a23 + a13 * s23);
    double p0 = a12 * (a12 * s23 - a23 * s12);
    p3 = 1.0 / p3;
    p2 = p2 * p3; p1 = p1 * p3; p0 = p0 * p3;
    const double g = p3p_cubic(p2, p1, p0);
    double A[9];
    A[0] = a23 * (1.0 - g);
    A[1] = (a23 * b12) * 0.5;
    A[2] = (a23 * b13 * g) * (-0.5);
    A[4] = a23 - a12 + a13 * g;
    A[5] = b23 * (a13 * g - a12) * 0.5;
    A[8] = g * (a13 - a23) - a12;
    A[3] = A[1]; A[6] = A[2]; A[7] = A[5];
    double V[9];
    jacobi_eig_n<3>(A, V, 8);
    // the eigenvalue of least magnitude is the known zero; e0 the larger of the other two in magnitude, e1 the smaller
    const double m0 = fabs(A[0]), m1 = fabs(A[4]), m2 = fabs(A[8]);
    int z = 0;
    if (m1 < m0) z = 1;
    if (m2 < (z == 0 ? m0 : m1)) z = 2;
    int e0 = z == 0 ? 1 : 0, e1 = z == 2 ? 1 : 2;
    const double me0 = e0 == 0 ? m0 : m1, me1 = e1 == 1 ? m1 : m2;
    if (me1 > me0) { const int tmp = e0; e0 = e1; e1 = tmp; }
    const double L0 = e0 == 0 ? A[0] : (e0 == 1 ? A[4] : A[8]);
    const double L1 = e1 == 0 ? A[0] : (e1 == 1 ? A[4] : A[8]);
    const double v = sqrt(fmax(0.0, -L1 / L0));
    double Ls[4][3];
    int n = 0;
    p3p_line(v, V, e0, e1, a12, a13, a23, b12, b13, b23, Ls, n);
    p3p_line(-v, V, e0, e1, a12, a13, a23, b12, b13, b23, Ls, n);
    // R = Y Xm^-1 with Xm = [d12 d13 d12xd13] (columns)
    const double cx0 = d12[1] * d13[2] - d12[2] * d13[1];
    const double cx1 = d12[2] * d13[0] - d12[0] * d13[2];
    const double cx2 = d12[0] * d13[1] - d12[1] * d13[0];
    const double m[9] = {d12[0], d13[0], cx0, d12[1], d13[1], cx1, d12[2], d13[2], cx2};
    double mi[9];
    {
        const double c00 = m[4] * m[8] - m[5] * m[7], c01 = m[5] * m[6] - m[3] * m[8], c02 = m[3] * m[7] - m[4] * m[6];
        const double id = 1.0 / (m[0] * c00 + m[1] * c01 + m[2] * c02);
        mi[0] = c00 * id; mi[1] = (m[2] * m[7] - m[1] * m[8]) * id; mi[2] = (m[1] * m[5] - m[2] * m[4]) * id;
        mi[3] = c01 * id; mi[4] = (m[0] * m[8] - m[2] * m[6]) * id; mi[5] = (m[2] * m[3] - m[0] * m[5]) * id;
        mi[6] = c02 * id; mi[7] = (m[1] * m[6] - m[0] * m[7]) * id; mi[8] = (m[0] * m[4] - m[1] * m[3]) * id;
    }
    int kept = 0;
#pragma unroll 1
    for (int r = 0; r < n && r < 4; ++r) {
        double L[3] = {Ls[r][0], Ls[r][1], Ls[r][2]};
        p3p_refine_depths(L, a12, a13, a23, b12, b13, b23);
        if (!(L[0] > 0.0) || !(L[1] > 0.0) || !(L[2] > 0.0) || !is_finite(L[0]) || !is_finite(L[1]) || !is_finite(L[2])) continue;
        double ry[3][3];
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int c = 0; c < 3; ++c) ry[k][c] = y[k][c] * L[k];
        double yd1[3], yd2[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            yd1[c] = ry[0][c] - ry[1][c];
            yd2[c] = ry[0][c] - ry[2][c];
        }
        const double yx0 = yd1[1] * yd2[2] - yd1[2] * yd2[1];
        const double yx1 = yd1[2] * yd2[0] - yd1[0] * yd2[2];
        const double yx2 = yd1[0] * yd2[1] - yd1[1] * yd2[0];
        const double Y[9] = {yd1[0], yd2[0], yx0, yd1[1], yd2[1], yx1, yd1[2], yd2[2], yx2};
        double P[12];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) P[3 * i + j] = Y[3 * i] * mi[j] + Y[3 * i + 1] * mi[3 + j] + Y[3 * i + 2] * mi[6 + j];
#pragma unroll
        for (int i = 0; i < 3; ++i) P[9 + i] = ry[0][i] - (P[3 * i] * X[0][0] + P[3 * i + 1] * X[0][1] + P[3 * i + 2] * X[0][2]);
        bool ok = true;
#pragma unroll
        for (int i = 0; i < 12; ++i) ok = ok && is_finite(P[i]);
        if (!ok) continue;
#pragma unroll
        for (int i = 0; i < 12; ++i) out[12 * kept + i] = P[i];
        ++kept;
    }
    return kept;
}

// ------------------------------------------------------------------------------------------------------------ RANSAC
struct PnpSmem {
    double pose[kBatch * kPnpRoots * 12];   // the batch's poses, 12 doubles per (hypothesis, root) slot
    double best[12];
    double part[kPnpSums * 8];              // block_tree_sum_many scratch
    double tot[kPnpSums];
    int nm[kBatch];
    int list[kBatch * kPnpRoots];
    int cnt[kBatch * kPnpRoots];
    int total, best_n, stop, scratch;
};

constexpr size_t pnp_smem_fixed() { return (sizeof(PnpSmem) + 15) & ~(size_t)15; }
static_assert(pnp_smem_fixed() + (size_t)kPnpCap * 40 + 1024 <= 228 * 1024, "the staged correspondences must fit one CTA's shared memory");

// Correspondence i of a query: staged (x^, y^) and X for i < cap, else computed from global memory with the same operations.
struct PnpPts {
    const double2* snxy;
    const double* sX;
    const float* gxy;
    const double* gX;
    double fx, fy, cx, cy;
    int cap;
    __device__ __forceinline__ void get(int i, double& x, double& y, double* Xw) const
    {
        if (i < cap) {
            const double2 v = snxy[i];
            x = v.x; y = v.y;
            Xw[0] = sX[3 * i]; Xw[1] = sX[3 * i + 1]; Xw[2] = sX[3 * i + 2];
        } else {
            x = ((double)__ldg(gxy + 2 * i) - cx) / fx;
            y = ((double)__ldg(gxy + 2 * i + 1) - cy) / fy;
            Xw[0] = __ldg(gX + 3ll * i); Xw[1] = __ldg(gX + 3ll * i + 1); Xw[2] = __ldg(gX + 3ll * i + 2);
        }
    }
};

static __device__ __forceinline__ void to_camera(const double* P, double fx, double fy, Camera& K)
{
    K.fx = fx; K.fy = fy;
#pragma unroll
    for (int i = 0; i < 9; ++i) K.r[i] = P[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) K.t[i] = P[9 + i];
}

// Inliers of pose K over the query, counted by the block (every thread returns the total); mask may be null.
static __device__ int block_count(const PnpPts& pts, int M, const Camera& K, double thr2, uint8_t* mask, int* scratch)
{
    int n = 0;
    for (int i = threadIdx.x; i < M; i += kRansacThreads) {
        double x, y, Xw[3], e2;
        pts.get(i, x, y, Xw);
        const bool in = reproject(K, Xw, x, y, thr2, e2);
        if (mask) mask[i] = (uint8_t)in;
        n += in;
    }
    for (int off = 16; off >= 1; off >>= 1) n += __shfl_down_sync(0xffffffffu, n, off);
    __syncthreads();
    if (threadIdx.x == 0) *scratch = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) atomicAdd(scratch, n);
    __syncthreads();
    const int total = *scratch;
    __syncthreads();
    return total;
}

// Adds one observation's Gauss-Newton terms at pose K: the upper triangle of J^T J (21, row by row, the u row's product then
// the v row's), J^T r (6) and the squared error, with J the rows of pose_rows (ransac_common.cuh).
static __device__ __forceinline__ void add_gn(double (&v)[kPnpSums], const Camera& K, double x, double y, const double* Xw)
{
    PoseRows J;
    pose_rows(K, x, y, Xw, J);
    const double ex = J.ex, ey = J.ey;
    const double(&ju)[6] = J.ju;
    const double(&jv)[6] = J.jv;
    int e = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = i; j < 6; ++j) {
            v[e] = v[e] + ju[i] * ju[j];
            v[e] = v[e] + jv[i] * jv[j];
            ++e;
        }
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        v[21 + i] = v[21 + i] + ju[i] * ex;
        v[21 + i] = v[21 + i] + jv[i] * ey;
    }
    v[27] = v[27] + (ex * ex + ey * ey);
}

// The Gauss-Newton step from the sums: Cholesky of J^T J, delta = -(J^T J)^-1 J^T r, applied by apply_pose_step
// (ransac_common.cuh).  False when a pivot is not positive.
static __device__ __forceinline__ bool gn_step(const double (&v)[kPnpSums], const Camera& K, Camera& O)
{
    double H[36];
    int e = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = i; j < 6; ++j) {
            H[i * 6 + j] = v[e];
            H[j * 6 + i] = v[e];
            ++e;
        }
    double L[36], inv[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        double s = H[j * 6 + j];
#pragma unroll
        for (int k = 0; k < j; ++k) s = s - L[j * 6 + k] * L[j * 6 + k];
        if (!(s > 0.0)) return false;
        const double d = sqrt(s);
        inv[j] = 1.0 / d;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            double w = H[i * 6 + j];
#pragma unroll
            for (int k = 0; k < j; ++k) w = w - L[i * 6 + k] * L[j * 6 + k];
            L[i * 6 + j] = w * inv[j];
        }
        L[j * 6 + j] = d;
    }
    double z[6], dl[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double w = -v[21 + i];
#pragma unroll
        for (int k = 0; k < i; ++k) w = w - L[i * 6 + k] * z[k];
        z[i] = w * inv[i];
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {
        double w = z[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) w = w - L[k * 6 + i] * dl[k];
        dl[i] = w * inv[i];
    }
    apply_pose_step(dl, K, O);
    return true;
}

__global__ void __launch_bounds__(kRansacThreads, 1) pnp_ransac_kernel(
    int n_images, const double* __restrict__ cams, const int32_t* __restrict__ image, const float* __restrict__ xy,
    const double* __restrict__ Xg, int stride, const int32_t* __restrict__ count, sfm_pnp_params prm, int cap,
    double* __restrict__ out_pose, int32_t* __restrict__ out_ninl, uint8_t* __restrict__ out_status, uint8_t* __restrict__ out_mask,
    int32_t* __restrict__ out_iters, unsigned long long* __restrict__ out_counts)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    PnpSmem& S = *reinterpret_cast<PnpSmem*>(smem_raw);
    double2* snxy = reinterpret_cast<double2*>(smem_raw + pnp_smem_fixed());
    double* sX = reinterpret_cast<double*>(snxy + cap);
    const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long base = (long long)q * stride;
    uint8_t* mask = out_mask + base;
    const double thr2 = prm.max_error * prm.max_error;

    const int img = __ldg(image + q);
    double fx = 0.0, fy = 0.0, cx = 0.0, cy = 0.0;
    int status = kPnpOk, M = 0;
    if (img < 0 || img >= n_images) {
        status = kPnpInvalid;
    } else {
        const double* c = cams + 16ll * img;
        fx = __ldg(c); fy = __ldg(c + 1); cx = __ldg(c + 2); cy = __ldg(c + 3);
        if (!(fx > 0.0) || !(fy > 0.0) || !is_finite(fx) || !is_finite(fy)) status = kPnpInvalid;
    }
    if (status == kPnpOk) {
        M = min(max(__ldg(count + q), 0), stride);
        if (M < 3) status = kPnpFew;
    }
    const float* gxy = xy + 2 * base;
    const double* gX = Xg + 3 * base;
    const PnpPts pts{snxy, sX, gxy, gX, fx, fy, cx, cy, cap};
    int cur = 0, done = 0;
    if (status == kPnpOk) {
        for (int i = tid; i < min(M, cap); i += kRansacThreads) {
            snxy[i] = make_double2(((double)__ldg(gxy + 2 * i) - cx) / fx, ((double)__ldg(gxy + 2 * i + 1) - cy) / fy);
            sX[3 * i] = __ldg(gX + 3ll * i); sX[3 * i + 1] = __ldg(gX + 3ll * i + 1); sX[3 * i + 2] = __ldg(gX + 3ll * i + 2);
        }
        if (tid == 0) S.best_n = -1;
        __syncthreads();
        // ---- search
        while (done < prm.max_iters) {
            const int nb = min(ransac_batch(done), prm.max_iters - done);
            if (tid < kBatch) {
                int n = 0;
                if (tid < nb) {
                    int idx[3];
                    draw_sample(prm.seed, (uint32_t)img, (uint32_t)(done + tid), 3, M, idx);
                    double nx[3], ny[3], Xs[3][3];
#pragma unroll
                    for (int k = 0; k < 3; ++k) pts.get(idx[k], nx[k], ny[k], Xs[k]);
                    n = p3p(nx, ny, Xs, S.pose + tid * kPnpRoots * 12);
                }
                S.nm[tid] = n;
            }
            __syncthreads();
            if (tid < kBatch) {
                int off = 0;
                for (int j = 0; j < tid; ++j) off += S.nm[j];
                for (int r = 0; r < S.nm[tid]; ++r) S.list[off + r] = tid * kPnpRoots + r;
                if (tid == kBatch - 1) S.total = off + S.nm[tid];
            }
            __syncthreads();
            const int total = S.total;
            for (int g = warp * kPnpGroup; g < total; g += (kRansacThreads / 32) * kPnpGroup) {
                Camera K[kPnpGroup];
                int c[kPnpGroup];
#pragma unroll
                for (int j = 0; j < kPnpGroup; ++j) {
                    to_camera(S.pose + S.list[min(g + j, total - 1)] * 12, fx, fy, K[j]);
                    c[j] = 0;
                }
                for (int i = lane; i < M; i += 32) {
                    double x, y, Xw[3], e2;
                    pts.get(i, x, y, Xw);
#pragma unroll
                    for (int j = 0; j < kPnpGroup; ++j) c[j] += reproject(K[j], Xw, x, y, thr2, e2);
                }
#pragma unroll
                for (int j = 0; j < kPnpGroup; ++j) {
                    int v = c[j];
                    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                    if (lane == 0 && g + j < total) S.cnt[g + j] = v;
                }
            }
            __syncthreads();
            if (tid == 0) {
                int best = S.best_n, arg = -1;
                for (int k = 0; k < total; ++k)
                    if (S.cnt[k] > best) { best = S.cnt[k]; arg = k; }
                if (arg >= 0) {
                    S.best_n = best;
                    for (int i = 0; i < 12; ++i) S.best[i] = S.pose[S.list[arg] * 12 + i];
                }
                S.stop = should_stop(S.best_n, M, 3, done + nb, prm.confidence) ? 1 : 0;
            }
            __syncthreads();
            done += nb;
            if (S.stop) break;
        }
        cur = S.best_n;
        if (cur < 0) {
            status = kPnpNoModel;
        } else {
            // ---- refine
            Camera P;
            to_camera(S.best, fx, fy, P);
            for (int round = 0; round < kLoRounds && prm.refine_iters > 0 && cur >= 3; ++round) {
                for (int i = tid; i < M; i += kRansacThreads) {         // the round's inliers (each thread reads back its own)
                    double x, y, Xw[3], e2;
                    pts.get(i, x, y, Xw);
                    mask[i] = (uint8_t)reproject(P, Xw, x, y, thr2, e2);
                }
                Camera it = P;
                bool moved = false;
                for (int s = 0; s < prm.refine_iters; ++s) {
                    double v[kPnpSums];
#pragma unroll
                    for (int e = 0; e < kPnpSums; ++e) v[e] = 0.0;
                    for (int i = tid; i < M; i += kRansacThreads)
                        if (mask[i]) {
                            double x, y, Xw[3];
                            pts.get(i, x, y, Xw);
                            add_gn(v, it, x, y, Xw);
                        }
                    block_tree_sum_many<kPnpSums>(v, S.part, S.tot);
                    Camera nx;
                    const bool ok = gn_step(v, it, nx);
                    double cost[1] = {0.0};
                    if (ok)
                        for (int i = tid; i < M; i += kRansacThreads)
                            if (mask[i]) {
                                double x, y, Xw[3], e2;
                                pts.get(i, x, y, Xw);
                                reproject(nx, Xw, x, y, thr2, e2);
                                cost[0] = cost[0] + e2;
                            }
                    __syncthreads();                                       // S.tot is rewritten below
                    if (!ok) break;
                    block_tree_sum_many<1>(cost, S.part, S.tot);
                    const bool better = cost[0] < v[27];
                    __syncthreads();
                    if (!better) break;
                    it = nx;
                    moved = true;
                }
                if (!moved) break;
                const int n = block_count(pts, M, it, thr2, nullptr, &S.scratch);
                if (n < cur) break;
                cur = n;
                P = it;
            }
            if (cur < prm.min_inliers || (double)cur < prm.min_inlier_ratio * (double)M) status = kPnpFewInliers;
            if (tid < 12) S.best[tid] = tid < 9 ? P.r[tid] : P.t[tid - 9];
            __syncthreads();
        }
    }
    // ---- emit
    if (status == kPnpOk) {
        Camera P;
        to_camera(S.best, fx, fy, P);
        for (int i = tid; i < stride; i += kRansacThreads) {
            uint8_t in = 0;
            if (i < M) {
                double x, y, Xw[3], e2;
                pts.get(i, x, y, Xw);
                in = (uint8_t)reproject(P, Xw, x, y, thr2, e2);
            }
            mask[i] = in;
        }
    } else {
        for (int i = tid; i < stride; i += kRansacThreads) mask[i] = 0;
    }
    if (tid < 12) out_pose[12ll * q + tid] = status == kPnpOk ? S.best[tid] : 0.0;
    if (tid == 0) {
        out_ninl[q] = (status == kPnpOk || status == kPnpFewInliers) ? cur : 0;
        out_status[q] = (uint8_t)status;
        if (out_iters) out_iters[q] = done;
        atomicAdd(&out_counts[status], 1ull);
    }
}

}  // namespace sfm

using namespace sfm;

extern "C" int sfm_pnp_gather(int n_images, int S, const int32_t* track_of, const int64_t* track_counts, int64_t max_tracks,
                              const uint8_t* point_status, const double* X, const float* xy, int xy_stride, const int32_t* image,
                              int n_query, float* out_xy, double* out_X, int32_t* out_feature, int32_t* out_count, void* stream)
{
    SFM_REQUIRE(n_query >= 0, "sfm_pnp_gather: negative query count");
    if (n_query == 0) return SFM_OK;
    SFM_REQUIRE(track_of && track_counts && point_status && X && xy && image && out_xy && out_X && out_feature && out_count,
                "sfm_pnp_gather: NULL argument");
    SFM_REQUIRE(n_images > 0 && S > 0, "sfm_pnp_gather: n_images and S must be positive");
    SFM_REQUIRE((long long)n_images * S < (1ll << 31), "sfm_pnp_gather: n_images * S = %lld must stay below 2^31", (long long)n_images * S);
    SFM_REQUIRE(xy_stride >= S, "sfm_pnp_gather: xy_stride %d is below S = %d", xy_stride, S);
    SFM_REQUIRE(max_tracks >= 0, "sfm_pnp_gather: negative track capacity");
    SFM_REQUIRE(((uintptr_t)xy & 7) == 0 && ((uintptr_t)out_xy & 7) == 0, "sfm_pnp_gather: xy and out_xy must be 8-byte aligned");
    pnp_gather_kernel<<<n_query, 256, 0, (cudaStream_t)stream>>>(n_images, S, track_of, track_counts, max_tracks, point_status, X, xy,
                                                                  xy_stride, image, out_xy, out_X, out_feature, out_count);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return SFM_OK;
}

extern "C" int sfm_pnp_ransac(int n_images, const double* cams, const int32_t* image, int n_query, const float* xy, const double* X,
                              int stride, const int32_t* count, const sfm_pnp_params* params, double* out_pose, int32_t* out_n_inliers,
                              uint8_t* out_status, uint8_t* out_mask, int32_t* out_iters, int64_t* out_counts, void* stream)
{
    SFM_REQUIRE(params, "sfm_pnp_ransac: NULL params");
    SFM_REQUIRE(out_counts && (n_query == 0 || (cams && image && xy && X && count && out_pose && out_n_inliers && out_status && out_mask)),
                "sfm_pnp_ransac: NULL argument");
    SFM_REQUIRE(n_images > 0 && stride > 0 && n_query >= 0, "sfm_pnp_ransac: n_images and stride must be positive, n_query non-negative");
    SFM_REQUIRE(params->max_iters > 0, "sfm_pnp_ransac: max_iters must be positive, got %d", params->max_iters);
    SFM_REQUIRE(params->min_inliers >= 3, "sfm_pnp_ransac: min_inliers must be at least 3, got %d", params->min_inliers);
    SFM_REQUIRE(params->min_inlier_ratio >= 0.0 && params->min_inlier_ratio <= 1.0, "sfm_pnp_ransac: min_inlier_ratio must lie in [0, 1], got %g",
                params->min_inlier_ratio);
    SFM_REQUIRE(params->refine_iters >= 0 && params->refine_iters <= 1000, "sfm_pnp_ransac: refine_iters must lie in [0, 1000], got %d",
                params->refine_iters);
    SFM_REQUIRE(params->max_error > 0.0 && params->max_error < 1e150, "sfm_pnp_ransac: max_error must be positive and finite, got %g",
                params->max_error);
    cudaStream_t st = (cudaStream_t)stream;
    SFM_CUDA_CHECK(cudaMemsetAsync(out_counts, 0, kPnpStatuses * sizeof(int64_t), st));
    if (n_query == 0) return SFM_OK;
    const int cap = std::min(stride, kPnpCap);
    const size_t smem = pnp_smem_fixed() + (size_t)cap * 40;
    static SmemAttrTable attr;
    SFM_CUDA_CHECK(ensure_dyn_smem(pnp_ransac_kernel, smem, current_device(), attr));
    pnp_ransac_kernel<<<n_query, kRansacThreads, smem, st>>>(n_images, cams, image, xy, X, stride, count, *params, cap, out_pose, out_n_inliers,
                                                              out_status, out_mask, out_iters, (unsigned long long*)out_counts);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return SFM_OK;
}
