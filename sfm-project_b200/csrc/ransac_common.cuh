// ransac_common.cuh -- the batched RANSAC driver that runs RANSAC-F (ransac_f.cu) and RANSAC-H (ransac_h.cu), and the
// numerical pieces those two and the pose kernel (pose.cu) share.  Every translation unit that includes this is compiled
// with -fmad=false: all floating-point work is IEEE basic arithmetic in a fixed order so that results are bit-identical
// to the C oracles under oracle/.
//
// ransac_driver<Model> is the whole kernel body: one CTA (256 threads) per image pair, correspondences staged once in
// shared memory as float4 (x1,y1,x2,y2), hypotheses in batches of 32, 32, 64, then 128 (ransac_batch):
//   solve   A: 8 lanes per minimal sample (one matrix row per lane, in registers): Hartley normalisation and the
//              Gauss-Jordan null space with complete pivoting (fp64, pivot search / row broadcast by shuffles)
//           B: one thread per sample turns its null space into up to Model::kRoots models
//   score   one warp per group of 4 models: every lane streams correspondences with 128-bit shared loads and scores
//           all 4 models (fp32, division-free), lane counts reduced with shuffles, exact bail-out
//   select  strict-greater argmax in (hypothesis, root) order, then the adaptive stop rule
// followed by an optional LO step (Hartley-normalised least-squares refit on the inliers, fixed-order fp64 reductions,
// smallest eigenvector of the 9 x 9 normal matrix) and the final mask.  The Model policy supplies only what depends on
// the model: sample size, the rows of phase A, phase B, the inlier predicate, the LO normal equations and the model
// made from the eigenvector (see FundamentalModel in ransac_f.cu, HomographyModel in ransac_h.cu).
#pragma once
#include <math.h>

#include <type_traits>

#include "common.cuh"

namespace sfm {

constexpr int kRansacThreads = 256;
constexpr int kBailEvery = 16;          // scoring: bail-out test every 16 warp iterations (512 correspondences)
constexpr int kBatch = 128;             // largest hypothesis batch
constexpr int kGroup = 4;               // models scored together by one warp
constexpr int kLoRounds = 2;
constexpr int kPtsCap = 4096;           // correspondences per pair staged in shared memory; wider pairs read the tail via L1/L2

// Hypotheses evaluated before the next termination check: 32, 32, 64, then 128 at a time (checks after 32, 64, 128, 256,
// 384, ... hypotheses).  Clean pairs -- the common case after the ratio test -- stop after the first 32.
__host__ __device__ constexpr int ransac_batch(int done) { return done < 64 ? 32 : (done < 128 ? 64 : 128); }

struct Norm2d { double s, cx, cy; };

// Correspondences of one pair: the first `cap` are staged in shared memory, the rest (very wide pairs only) are read
// through L1/L2.  Values are identical either way, so results do not depend on `cap`.
struct Pts {
    const float4* s;
    const float4* g;
    int cap;
    __device__ __forceinline__ float4 operator[](int i) const { return i < cap ? s[i] : __ldg(g + i); }
};

static __device__ __forceinline__ uint32_t rng_u32(uint64_t seed, uint32_t pair, uint32_t hyp, uint32_t ctr)
{
    uint64_t x = seed + 0x9E3779B97F4A7C15ULL * ((((uint64_t)pair) << 32) | (uint64_t)hyp);
    x ^= 0xD1B54A32D192ED03ULL * (uint64_t)(ctr + 1u);
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ULL;
    x ^= x >> 27; x *= 0x94D049BB133111EBULL;
    x ^= x >> 31;
    return (uint32_t)(x >> 32);
}

static __device__ void draw_sample(uint64_t seed, uint32_t pair, uint32_t hyp, int m, int M, int* idx)
{
    for (int k = 0; k < m; ++k) {
        int v = 0;
        for (int attempt = 0; attempt < 16; ++attempt) {
            const uint32_t r = rng_u32(seed, pair, hyp, (uint32_t)(k * 16 + attempt));
            v = (int)(((uint64_t)r * (uint64_t)(uint32_t)M) >> 32);
            int dup = 0;
            for (int j = 0; j < k; ++j) dup |= (idx[j] == v);
            if (!dup) break;
        }
        idx[k] = v;
    }
}

// The m correspondence indices of hypothesis `hyp`: the caller's `samples` rows ([max_iters, 8], reduced mod M) or drawn
static __device__ __forceinline__ void hypothesis_sample(const uint32_t* samples, uint64_t seed, uint32_t pair, int hyp, int m,
                                                         int M, int* idx)
{
    if (samples) {
        for (int k = 0; k < m; ++k) idx[k] = (int)(samples[(size_t)hyp * 8 + k] % (uint32_t)M);
    } else {
        draw_sample(seed, pair, (uint32_t)hyp, m, M, idx);
    }
}

// Phase A's Hartley normalisation of a K-point sample (every lane of the octet computes the same values) and the
// normalised coordinates (u1, v1, u2, v2) of sample point k.  False when the points of either image coincide.
template <int K>
static __device__ __forceinline__ bool hartley_sample(const Pts& pts, const int* idx, int k, Norm2d& n1, Norm2d& n2, double& u1,
                                                      double& v1, double& u2, double& v2)
{
    double x1[K], y1[K], x2[K], y2[K];
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const float4 c = pts[idx[j]];
        x1[j] = (double)c.x; y1[j] = (double)c.y; x2[j] = (double)c.z; y2[j] = (double)c.w;
    }
    double sx = 0.0, sy = 0.0, tx = 0.0, ty = 0.0;
#pragma unroll
    for (int j = 0; j < K; ++j) { sx += x1[j]; sy += y1[j]; tx += x2[j]; ty += y2[j]; }
    const double inv = 1.0 / (double)K;
    n1.cx = sx * inv; n1.cy = sy * inv; n2.cx = tx * inv; n2.cy = ty * inv;
    double d1 = 0.0, d2 = 0.0;
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const double ax = x1[j] - n1.cx, ay = y1[j] - n1.cy;
        const double bx = x2[j] - n2.cx, by = y2[j] - n2.cy;
        d1 += sqrt(ax * ax + ay * ay);
        d2 += sqrt(bx * bx + by * by);
    }
    d1 *= inv; d2 *= inv;
    if (!(d1 > 1e-9) || !(d2 > 1e-9)) return false;
    n1.s = 1.4142135623730951 / d1;
    n2.s = 1.4142135623730951 / d2;
    double mx1 = x1[0], my1 = y1[0], mx2 = x2[0], my2 = y2[0];
#pragma unroll
    for (int j = 1; j < K; ++j)
        if (k == j) { mx1 = x1[j]; my1 = y1[j]; mx2 = x2[j]; my2 = y2[j]; }
    u1 = (mx1 - n1.cx) * n1.s; v1 = (my1 - n1.cy) * n1.s;
    u2 = (mx2 - n2.cx) * n2.s; v2 = (my2 - n2.cy) * n2.s;
    return true;
}

// The two normalisations travel from phase A to phase B in doubles 18..23 of a hypothesis' 24-double slot
static __device__ __forceinline__ void store_norms(double* out, const Norm2d& n1, const Norm2d& n2)
{
    out[18] = n1.s; out[19] = n1.cx; out[20] = n1.cy;
    out[21] = n2.s; out[22] = n2.cx; out[23] = n2.cy;
}

static __device__ __forceinline__ void load_norms(const double* in, Norm2d& n1, Norm2d& n2)
{
    n1.s = in[18]; n1.cx = in[19]; n1.cy = in[20];
    n2.s = in[21]; n2.cx = in[22]; n2.cy = in[23];
}

// Cyclic Jacobi on a symmetric N x N matrix: A diagonal -> eigenvalues, V columns -> eigenvectors.  The dimension is
// known at compile time, so every index is static and A and V live in registers.
template <int N>
static __device__ __forceinline__ void jacobi_eig_n(double (&A)[N * N], double (&V)[N * N], int sweeps)
{
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) V[i * N + j] = (i == j) ? 1.0 : 0.0;
#pragma unroll 1
    for (int s = 0; s < sweeps; ++s) {
#pragma unroll
        for (int p = 0; p < N - 1; ++p) {
#pragma unroll
            for (int q = p + 1; q < N; ++q) {
                const double apq = A[p * N + q];
                if (apq == 0.0) continue;
                const double app = A[p * N + p], aqq = A[q * N + q];
                const double theta = (aqq - app) / (2.0 * apq);
                const double at = fabs(theta);
                double t = 1.0 / (at + sqrt(theta * theta + 1.0));
                if (theta < 0.0) t = -t;
                const double c = 1.0 / sqrt(t * t + 1.0);
                const double sn = t * c;
#pragma unroll
                for (int k = 0; k < N; ++k) {
                    const double akp = A[k * N + p], akq = A[k * N + q];
                    A[k * N + p] = c * akp - sn * akq;
                    A[k * N + q] = sn * akp + c * akq;
                }
#pragma unroll
                for (int k = 0; k < N; ++k) {
                    const double apk = A[p * N + k], aqk = A[q * N + k];
                    A[p * N + k] = c * apk - sn * aqk;
                    A[q * N + k] = sn * apk + c * aqk;
                }
#pragma unroll
                for (int k = 0; k < N; ++k) {
                    const double vkp = V[k * N + p], vkq = V[k * N + q];
                    V[k * N + p] = c * vkp - sn * vkq;
                    V[k * N + q] = sn * vkp + c * vkq;
                }
            }
        }
    }
}

// N block sums at once with ONE barrier pair (the LO refit needs 5 + 2 + 45 of them per round).  Each sum is a shfl_down
// tree per warp, then the eight warp sums added in warp order (oracle: lane_tree).  part: N * 8 doubles, tot: N doubles (shared memory); every thread returns with v[e] = the block total.
template <int N>
static __device__ __forceinline__ void block_tree_sum_many(double (&v)[N], double* part, double* tot)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int e = 0; e < N; ++e) {
        double x = v[e];
        for (int off = 16; off >= 1; off >>= 1) x += __shfl_down_sync(0xffffffffu, x, off);
        if (lane == 0) part[e * 8 + warp] = x;
    }
    __syncthreads();
    if (threadIdx.x < N) {
        double t = part[threadIdx.x * 8];
        for (int w = 1; w < kRansacThreads / 32; ++w) t += part[threadIdx.x * 8 + w];
        tot[threadIdx.x] = t;
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < N; ++e) v[e] = tot[e];
}

// Eigenvector of the smallest eigenvalue of a symmetric positive semi-definite 9 x 9 matrix (the normal matrix of a
// DLT / 8-point system): Cholesky factor of A + eps*I (eps = 1e-13 * trace keeps exact data factorisable and does not
// move the eigenvectors), then inverse iterations from a fixed start vector until the normalised iterate stops moving
// (at most 16; well-conditioned systems take 3-4).  Serial, a few thousand cycles --
// the 10-sweep cyclic Jacobi it replaces took ~900 K cycles on one thread and made the LO refit 13x the cost of the
// whole hypothesis loop.  `w` is scratch for 45 doubles (shared memory).  Returns 0 when A is not usable.
static __device__ int smallest_eigvec9(const double* __restrict__ A, double* __restrict__ w, double* __restrict__ xout)
{
    double* __restrict__ L = w;            // packed lower triangle in shared memory, row i at L[i*(i+1)/2]
    double invd[9], x[9], y[9];            // statically indexed (every loop below is fully unrolled): registers
    double tr = 0.0;
#pragma unroll
    for (int i = 0; i < 9; ++i) tr += A[i * 9 + i];
    if (!(tr > 0.0) || !(tr < 1e300)) return 0;
    const double eps = tr * 1e-13;
#pragma unroll
    for (int j = 0; j < 9; ++j) {
        double sj = A[j * 9 + j] + eps;
#pragma unroll
        for (int k = 0; k < j; ++k) sj -= L[j * (j + 1) / 2 + k] * L[j * (j + 1) / 2 + k];
        if (!(sj > 0.0)) return 0;
        const double d = sqrt(sj);
        L[j * (j + 1) / 2 + j] = d;
        invd[j] = 1.0 / d;
#pragma unroll
        for (int i = j + 1; i < 9; ++i) {
            double v = A[i * 9 + j];
#pragma unroll
            for (int k = 0; k < j; ++k) v -= L[i * (i + 1) / 2 + k] * L[j * (j + 1) / 2 + k];
            L[i * (i + 1) / 2 + j] = v * invd[j];
        }
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) x[i] = 1.0 + 0.125 * (double)i;
#pragma unroll 1
    for (int it = 0; it < 16; ++it) {
#pragma unroll
        for (int i = 0; i < 9; ++i) {                       // L y = x
            double v = x[i];
#pragma unroll
            for (int k = 0; k < i; ++k) v -= L[i * (i + 1) / 2 + k] * y[k];
            y[i] = v * invd[i];
        }
        double z[9];
#pragma unroll
        for (int i = 8; i >= 0; --i) {                      // L^T z = y
            double v = y[i];
#pragma unroll
            for (int k = i + 1; k < 9; ++k) v -= L[k * (k + 1) / 2 + i] * z[k];
            z[i] = v * invd[i];
        }
        double ss = 0.0;
#pragma unroll
        for (int i = 0; i < 9; ++i) ss += z[i] * z[i];
        if (!(ss > 0.0) || !(ss < 1e300)) return 0;
        const double inv = 1.0 / sqrt(ss);
        double diff = 0.0;                                  // converged when the normalised iterate stops moving
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            const double xi = z[i] * inv;
            diff = fmax(diff, fabs(xi - x[i]));
            x[i] = xi;
        }
        if (it > 0 && diff < 1e-13) break;
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) xout[i] = x[i];
    return 1;
}

static __device__ bool should_stop(int best, int M, int m, int done, double confidence)
{
    if (confidence >= 1.0 || best <= 0) return false;
    const double w = (double)best / (double)M;
    double wm = 1.0;
    for (int k = 0; k < m; ++k) wm *= w;
    const double q = 1.0 - wm;
    if (!(q > 0.0)) return true;
    double res = 1.0, base = q;
    int e = done;
    while (e) { if (e & 1) res *= base; base *= base; e >>= 1; }
    return res <= (1.0 - confidence);
}

// A calibrated camera x ~ K (R X + t) with K's focal lengths; the principal point is applied to the observations instead
// (normalised coordinates x^ = (x - cx) / fx).  Shared by track triangulation (triangulate.cu) and registration (pnp.cu).
struct Camera {
    double fx, fy, r[9], t[3];
};

// One row of a [n, 16] camera table: fx fy cx cy, R (row-major), t
static __device__ __forceinline__ void load_camera(const double* __restrict__ c, Camera& K)
{
    K.fx = __ldg(c + 0);
    K.fy = __ldg(c + 1);
#pragma unroll
    for (int i = 0; i < 9; ++i) K.r[i] = __ldg(c + 4 + i);
#pragma unroll
    for (int i = 0; i < 3; ++i) K.t[i] = __ldg(c + 13 + i);
}

// Squared pixel reprojection error (e2 = +inf behind the camera); inlier iff in front and e2 <= thr2.  A triangulated point
// and a registered pose agree on what an inlier observation is because both use this predicate.
static __device__ __forceinline__ bool reproject(const Camera& K, const double* X, double x, double y, double thr2, double& e2)
{
    const double p0 = K.r[0] * X[0] + K.r[1] * X[1] + K.r[2] * X[2] + K.t[0];
    const double p1 = K.r[3] * X[0] + K.r[4] * X[1] + K.r[5] * X[2] + K.t[1];
    const double p2 = K.r[6] * X[0] + K.r[7] * X[1] + K.r[8] * X[2] + K.t[2];
    if (!(p2 > 0.0)) {
        e2 = __longlong_as_double(0x7ff0000000000000ll);
        return false;
    }
    const double iz = 1.0 / p2;
    const double ex = (p0 * iz - x) * K.fx;
    const double ey = (p1 * iz - y) * K.fy;
    e2 = ex * ex + ey * ey;
    return e2 <= thr2;
}

// Camera centre C = -R^T t
static __device__ __forceinline__ void camera_center(const Camera& K, double* C)
{
#pragma unroll
    for (int i = 0; i < 3; ++i) C[i] = -(K.r[i] * K.t[0] + K.r[3 + i] * K.t[1] + K.r[6 + i] * K.t[2]);
}

// cos of the angle at X between the rays from the centres Ca and Cb: the triangulation angle.  Track triangulation
// (triangulate.cu) keeps a hypothesis and the point filter (mapper.cu) keeps a point only when some pair of its views has
// ray_cos <= cos(min_angle); both use this one sequence of operations, so they agree to the bit.  Symmetric in a and b.
static __device__ __forceinline__ double ray_cos(const double* X, const double* Ca, const double* Cb)
{
    const double da0 = X[0] - Ca[0], da1 = X[1] - Ca[1], da2 = X[2] - Ca[2];
    const double db0 = X[0] - Cb[0], db1 = X[1] - Cb[1], db2 = X[2] - Cb[2];
    const double dot = da0 * db0 + da1 * db1 + da2 * db2;
    const double na = da0 * da0 + da1 * da1 + da2 * da2;
    const double nb = db0 * db0 + db1 * db1 + db2 * db2;
    return dot / sqrt(na * nb);
}

// The pixel residual of one observation (x^, y^) of Xw at pose K and its Jacobian rows for the camera-frame perturbation
// R' = dR(w) R, t' = dR(w) t + dt, taken at p = R X + t: its linearisation error scales with the depth, not with |X|, so a
// step still lowers the cost when the world is far from its origin.  Shared by registration (pnp.cu) and bundle
// adjustment (bundle.cu); d(u, v) / dp is (a0, 0, a2) and (0, b1, b2), so d(u, v) / dX is that times R.
struct PoseRows {
    double p0, p1, p2;
    double a0, a2, b1, b2;
    double ex, ey;
    double ju[6], jv[6];                // d(u, v) / d(w, t)
};

static __device__ __forceinline__ void pose_rows(const Camera& K, double x, double y, const double* Xw, PoseRows& J)
{
    const double q0 = K.r[0] * Xw[0] + K.r[1] * Xw[1] + K.r[2] * Xw[2];
    const double q1 = K.r[3] * Xw[0] + K.r[4] * Xw[1] + K.r[5] * Xw[2];
    const double q2 = K.r[6] * Xw[0] + K.r[7] * Xw[1] + K.r[8] * Xw[2];
    const double p0 = q0 + K.t[0], p1 = q1 + K.t[1], p2 = q2 + K.t[2];
    const double iz = 1.0 / p2;
    const double u0 = p0 * iz, u1 = p1 * iz;
    J.p0 = p0; J.p1 = p1; J.p2 = p2;
    J.ex = (u0 - x) * K.fx;
    J.ey = (u1 - y) * K.fy;
    J.a0 = K.fx * iz; J.a2 = -(J.a0 * u0);
    J.b1 = K.fy * iz; J.b2 = -(J.b1 * u1);
    J.ju[0] = J.a2 * p1; J.ju[1] = J.a0 * p2 - J.a2 * p0; J.ju[2] = -(J.a0 * p1); J.ju[3] = J.a0; J.ju[4] = 0.0; J.ju[5] = J.a2;
    J.jv[0] = J.b2 * p1 - J.b1 * p2; J.jv[1] = -(J.b2 * p0); J.jv[2] = J.b1 * p0; J.jv[3] = 0.0; J.jv[4] = J.b1; J.jv[5] = J.b2;
}

// The pose after the step dl = (w, dt) of that perturbation: R' = dR R with dR the rotation of the normalised quaternion
// (1, w/2), t' = dR t + dt.
static __device__ __forceinline__ void apply_pose_step(const double* dl, const Camera& K, Camera& O)
{
    const double hx = 0.5 * dl[0], hy = 0.5 * dl[1], hz = 0.5 * dl[2];
    const double in = 1.0 / sqrt(1.0 + hx * hx + hy * hy + hz * hz);
    const double qw = in, qx = hx * in, qy = hy * in, qz = hz * in;
    const double D[9] = {1.0 - 2.0 * (qy * qy + qz * qz), 2.0 * (qx * qy - qw * qz), 2.0 * (qx * qz + qw * qy),
                         2.0 * (qx * qy + qw * qz), 1.0 - 2.0 * (qx * qx + qz * qz), 2.0 * (qy * qz - qw * qx),
                         2.0 * (qx * qz - qw * qy), 2.0 * (qy * qz + qw * qx), 1.0 - 2.0 * (qx * qx + qy * qy)};
    O.fx = K.fx; O.fy = K.fy;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) O.r[3 * i + j] = D[3 * i] * K.r[j] + D[3 * i + 1] * K.r[3 + j] + D[3 * i + 2] * K.r[6 + j];
#pragma unroll
    for (int i = 0; i < 3; ++i) O.t[i] = (D[3 * i] * K.t[0] + D[3 * i + 1] * K.t[1] + D[3 * i + 2] * K.t[2]) + dl[3 + i];
}

// ---------------------------------------------------------------------------------------------------------------
// Cooperative Gauss-Jordan elimination with complete pivoting: 8 lanes (one aligned octet of a warp) reduce ONE
// m x 9 system, lane r holding row r in registers (a[0..8], statically indexed).  Value for value the serial
// elimination of oracle/ransac_f.c / ransac_h.c: rows and columns are never moved, their LOGICAL positions are
// tracked instead (lrow per lane; lc / pc = logical<->physical column maps, 4 bits per entry), the pivot search
// breaks ties by the smallest logical (row, column) exactly like the serial strict-greater scan, and every element
// sees the same operations (a *= 1/pivot on the pivot row, a -= f * pivot_row elsewhere) in the same order.
// The serial version keeps 8x9 doubles per thread in local memory, which thrashes L1 at 2 CTAs / SM; this one
// keeps 18 registers per lane and uses all 256 threads of the CTA.
struct CoopGJ {
    unsigned long long lc;   // lc[j]: logical position of physical column j
    unsigned long long pc;   // pc[k]: physical column at logical position k
    int lrow;                // logical position of this lane's row (15 = lane holds no row)
};

static __device__ __forceinline__ double sel9(const double (&a)[9], int i)
{
    double v = a[0];
#pragma unroll
    for (int j = 1; j < 9; ++j) v = (i == j) ? a[j] : v;
    return v;
}

static __device__ __forceinline__ unsigned long long set4(unsigned long long w, int pos, int val)
{
    return (w & ~(15ull << (4 * pos))) | ((unsigned long long)val << (4 * pos));
}

// Returns false (in every lane of the octet) when a pivot is <= tol.  On success st describes the final layout.
template <int M>
static __device__ __forceinline__ bool coop_gauss_jordan(double (&a)[9], int sl, unsigned gmask, double tol, CoopGJ& st)
{
    st.lc = 0x876543210ull;
    st.pc = 0x876543210ull;
    st.lrow = (sl < M) ? sl : 15;
    const int src0 = (threadIdx.x & 24);                     // first lane of this octet within the warp
#pragma unroll 1
    for (int k = 0; k < M; ++k) {
        double bv = -1.0;
        int bkey = 0x7fffffff;
        if (st.lrow != 15 && st.lrow >= k) {
#pragma unroll
            for (int j = 0; j < 9; ++j) {
                const int lj = (int)(st.lc >> (4 * j)) & 15;
                const double v = fabs(a[j]);
                const int key = ((st.lrow * 9 + lj) << 8) | (sl << 4) | j;
                if (lj >= k && (v > bv || (v == bv && key < bkey))) { bv = v; bkey = key; }
            }
        }
#pragma unroll
        for (int o = 1; o <= 4; o <<= 1) {
            const double ov = __shfl_xor_sync(gmask, bv, o);
            const int ok = __shfl_xor_sync(gmask, bkey, o);
            if (ov > bv || (ov == bv && ok < bkey)) { bv = ov; bkey = ok; }
        }
        if (!(bv > tol)) return false;
        const int pl = (bkey >> 4) & 15, pcol = bkey & 15;
        const int lidx = bkey >> 8, pi = lidx / 9, pj = lidx - 9 * pi;
        if (st.lrow == k) st.lrow = pi;
        else if (sl == pl) st.lrow = k;
        const int c0 = (int)(st.pc >> (4 * k)) & 15;          // physical column now at logical k moves to logical pj
        st.lc = set4(set4(st.lc, c0, pj), pcol, k);
        st.pc = set4(set4(st.pc, pj, c0), k, pcol);
        const double own = sel9(a, pcol);                     // pivot lane: the pivot; other lanes: their factor f
        if (sl == pl) {
            const double inv = 1.0 / own;
#pragma unroll
            for (int j = 0; j < 9; ++j)
                if (((int)(st.lc >> (4 * j)) & 15) >= k) a[j] *= inv;
        }
        double r[9];
#pragma unroll
        for (int j = 0; j < 9; ++j) r[j] = __shfl_sync(gmask, a[j], src0 + pl);
        if (sl != pl && sl < M) {
#pragma unroll
            for (int j = 0; j < 9; ++j)
                if (((int)(st.lc >> (4 * j)) & 15) >= k) a[j] -= own * r[j];
        }
    }
    return true;
}

// After a successful elimination: scatter null vector c (c < 9 - M) into dst[0..8] (shared memory, one writer per entry).
template <int M>
static __device__ __forceinline__ void coop_null_vector(const double (&a)[9], int sl, const CoopGJ& st, int c, double* dst)
{
    const int fc = (int)(st.pc >> (4 * (M + c))) & 15;        // physical free column of this null vector
    if (sl < M) dst[(int)(st.pc >> (4 * st.lrow)) & 15] = -sel9(a, fc);
    if (sl == 0) {
#pragma unroll
        for (int e = 0; e < 9 - M; ++e) dst[(int)(st.pc >> (4 * (M + e))) & 15] = (e == c) ? 1.0 : 0.0;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// The RANSAC driver.  Model is a policy struct:
//   kMaxSample, kRoots        largest sample size; models per hypothesis (model-list entry = hypothesis * kRoots + root)
//   kLoMin                    fewest inliers the LO refit runs on
//   kSampleInPhaseB           phase B needs the sample indices again
//   check(prm)                host: checks of the parameter fields only this model reads
//   sample_size(prm)          m
//   null_space(pts, idx, m, sl, gmask, out)      phase A for one octet: null space(s) in out[0..17], normalisations in out[18..23]
//   models(in, m, pts, idx, out)                 phase B: up to kRoots unit-norm models from one slot; returns their number
//   inlier(model, c, thr2, score)                fp32 inlier predicate
//   lo_rows(acc, u1, v1, u2, v2)                 adds one inlier's rows to the 45 upper-triangle entries of the normal matrix
//   refit(h, n1, n2, out)                        model from the smallest eigenvector h (normalised frame); 0 when unusable
template <class Model>
struct RansacSmem {
    // phase A -> B: 24 doubles per hypothesis; then the models (9 doubles each); in LO, the eigen-problem and reductions
    double modelD[kBatch * 24 > kBatch * Model::kRoots * 9 ? kBatch * 24 : kBatch * Model::kRoots * 9];
    double bestM[9];
    double trialM[9];
    float modelF[kBatch * Model::kRoots * 9];
    int nm[kBatch];
    int list[kBatch * Model::kRoots];
    int cnt[kBatch * Model::kRoots];
    int total, best, stop, ok;
};

template <class Model>
constexpr size_t ransac_smem_fixed() { return (sizeof(RansacSmem<Model>) + 15) & ~(size_t)15; }

template <class Model>
static __device__ int block_count_inliers(const double* Md, const Pts& pts, int M, float thr2, int score,
                                          uint8_t* __restrict__ mask, int* scratch)
{
    float F[9];
    for (int i = 0; i < 9; ++i) F[i] = (float)Md[i];
    int n = 0;
    for (int i = threadIdx.x; i < M; i += kRansacThreads) {
        const bool in = Model::inlier(F, pts[i], thr2, score);
        if (mask) mask[i] = (uint8_t)in;
        n += in;
    }
    for (int off = 16; off >= 1; off >>= 1) n += __shfl_down_sync(0xffffffffu, n, off);
    __syncthreads();
    if (threadIdx.x == 0) *scratch = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) atomicAdd(scratch, n);
    __syncthreads();
    return *scratch;
}

// One CTA per pair.  stop_target (may be null): sampling ends once a model with max(best, target) inliers would have been
// found with the requested confidence.
template <class Model>
static __device__ __forceinline__ void ransac_driver(
    const float* __restrict__ corr, int corr_stride, const int32_t* __restrict__ count, const int32_t* __restrict__ offsets,
    const uint32_t* __restrict__ pair_id, const uint32_t* __restrict__ samples, const int32_t* __restrict__ stop_target,
    sfm_ransac_params prm, int pts_cap, double* __restrict__ out_model, int32_t* __restrict__ out_ninl,
    uint8_t* __restrict__ out_mask, int32_t* __restrict__ out_iters)
{
    // two CTAs per SM (DESIGN §4): fixed part + staged points + the 1 KB the hardware reserves per CTA
    static_assert(2 * (ransac_smem_fixed<Model>() + kPtsCap * 16 + 1024) <= 228 * 1024, "two RANSAC CTAs must fit on one SM");
    constexpr int kRoots = Model::kRoots;
    extern __shared__ __align__(16) uint8_t smem_raw[];
    RansacSmem<Model>& S = *reinterpret_cast<RansacSmem<Model>*>(smem_raw);
    float4* spts = reinterpret_cast<float4*>(smem_raw + ransac_smem_fixed<Model>());

    const int p = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // strided layout: pair p owns rows [p * corr_stride, +count[p]); packed layout: rows [offsets[p], offsets[p+1])
    const long long base = offsets ? (long long)offsets[p] : (long long)p * corr_stride;
    const int M = offsets ? (offsets[p + 1] - offsets[p]) : min(count[p], corr_stride);
    const int m = Model::sample_size(prm);
    const float thr2 = prm.threshold * prm.threshold;
    uint8_t* mask = out_mask + base;
    const float4* gpts = reinterpret_cast<const float4*>(corr) + base;

    for (int i = tid; i < (offsets ? M : corr_stride); i += kRansacThreads) mask[i] = 0;
    if (tid < 9) out_model[(long long)p * 9 + tid] = 0.0;
    if (tid == 0) { out_ninl[p] = 0; if (out_iters) out_iters[p] = 0; S.best = 0; S.stop = 0; }
    if (M < m) return;

    for (int i = tid; i < min(M, pts_cap); i += kRansacThreads) spts[i] = gpts[i];
    const Pts pts{spts, gpts, pts_cap};
    const uint32_t pid = pair_id ? pair_id[p] : (uint32_t)p;
    const int target = stop_target ? min(max(stop_target[p], 0), M) : 0;
    __syncthreads();

    int done = 0;
    while (done < prm.max_iters) {
        const int nb = min(ransac_batch(done), prm.max_iters - done);
        // ---- solve, phase A: 8 lanes per hypothesis -> null spaces in shared memory (S.modelD, 24 doubles each)
        {
            const int sl = tid & 7;
            const unsigned gmask = 0xFFu << (lane & 24);
            for (int h = tid >> 3; h < kBatch; h += kRansacThreads / 8) {
                bool ok = false;
                if (h < nb) {
                    int idx[Model::kMaxSample];
                    hypothesis_sample(samples, prm.seed, pid, done + h, m, M, idx);
                    ok = Model::null_space(pts, idx, m, sl, gmask, S.modelD + h * 24);
                }
                if (sl == 0) S.nm[h] = ok ? 1 : 0;
            }
        }
        __syncthreads();
        // ---- solve, phase B: one thread per hypothesis finishes its models in registers; after the barrier they overwrite
        // the null spaces
        {
            double Mm[9 * kRoots];
            int n = 0;
            if (tid < kBatch && S.nm[tid]) {
                int idx[Model::kMaxSample];
                if constexpr (Model::kSampleInPhaseB) hypothesis_sample(samples, prm.seed, pid, done + tid, m, M, idx);
                n = Model::models(S.modelD + tid * 24, m, pts, idx, Mm);
            }
            __syncthreads();
            if (tid < kBatch) {
                for (int r = 0; r < n; ++r)
                    for (int i = 0; i < 9; ++i) {
                        S.modelD[(tid * kRoots + r) * 9 + i] = Mm[9 * r + i];
                        S.modelF[(tid * kRoots + r) * 9 + i] = (float)Mm[9 * r + i];
                    }
                S.nm[tid] = n;
            }
        }
        __syncthreads();
        if (tid < kBatch) {
            int off = 0;
            for (int j = 0; j < tid; ++j) off += S.nm[j];
            for (int r = 0; r < S.nm[tid]; ++r) S.list[off + r] = tid * kRoots + r;
            if (tid == kBatch - 1) S.total = off + S.nm[tid];
        }
        __syncthreads();
        // ---- score: a warp takes 4 models at a time and streams every correspondence once for all of them
        const int total = S.total;
        for (int g = warp * kGroup; g < total; g += (kRansacThreads / 32) * kGroup) {
            float F[kGroup][9];
            int c[kGroup];
#pragma unroll
            for (int j = 0; j < kGroup; ++j) {
                const int slot = S.list[min(g + j, total - 1)];
#pragma unroll
                for (int i = 0; i < 9; ++i) F[j][i] = S.modelF[slot * 9 + i];
                c[j] = 0;
            }
            // the next correspondence is loaded before the current one is scored: the shared-memory latency hides behind
            // the ~100 arithmetic instructions of the four models
            float4 nx = pts[min(lane, M - 1)];
            // exact bail-out: once none of the four models can still EXCEED the best count of the earlier batches (their
            // counts so far + every correspondence not yet seen), the rest of the stream is skipped.  The partial counts stay
            // <= that best, so the strict-greater selection -- and therefore the result -- is unchanged.
            const int best_prev = S.best;
            const bool can_bail = best_prev * 4 > M;
            auto stream = [&](auto bail_c) {
                constexpr bool kBail = decltype(bail_c)::value;
                int next_check = lane + 32 * kBailEvery;
                for (int i = lane; i < M; i += 32) {
                    const float4 pt = nx;
                    nx = pts[min(i + 32, M - 1)];
#pragma unroll
                    for (int j = 0; j < kGroup; ++j) c[j] += Model::inlier(F[j], pt, thr2, prm.score);
                    if (kBail && i + 32 == next_check) {
                        next_check += 32 * kBailEvery;
                        const int left = M - (i - lane + 32);               // correspondences no lane has looked at yet
                        if (left <= 0) return;                               // (uniform: every lane was active in this iteration iff left >= 0)
                        int top = 0;
#pragma unroll
                        for (int j = 0; j < kGroup; ++j) {
                            int v = c[j];
                            for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                            top = max(top, v);
                        }
                        if (top + left <= best_prev) return;
                    }
                }
            };
            if (can_bail) stream(std::true_type{}); else stream(std::false_type{});      // no bail-out code in the common first batches
#pragma unroll
            for (int j = 0; j < kGroup; ++j) {
                int v = c[j];
                for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                if (lane == 0 && g + j < total) S.cnt[g + j] = v;
            }
        }
        __syncthreads();
        // ---- select (strict >, list order = (hypothesis, root) ascending) and stop rule
        if (tid == 0) {
            int best = S.best, arg = -1;
            for (int k = 0; k < total; ++k)
                if (S.cnt[k] > best) { best = S.cnt[k]; arg = k; }
            if (arg >= 0) {
                S.best = best;
                for (int i = 0; i < 9; ++i) S.bestM[i] = S.modelD[S.list[arg] * 9 + i];
            }
            S.stop = should_stop(max(S.best, target), M, m, done + nb, prm.confidence) ? 1 : 0;
        }
        __syncthreads();
        done += nb;
        if (S.stop) break;
    }
    if (tid == 0 && out_iters) out_iters[p] = done;
    if (S.best < m) return;                 // fewer inliers than the sample size: no model

    int best = block_count_inliers<Model>(S.bestM, pts, M, thr2, prm.score, mask, &S.total);
    if (prm.lo_refit) {
        for (int round = 0; round < kLoRounds; ++round) {
            __syncthreads();
            // moments of the inliers (fixed lane order)
            double* red_part = S.modelD + 256;   // scratch of the batched reductions: 45 * 8 partials + 45 totals (AtA and the
            double* red_tot = red_part + 45 * 8;  // eigen-solver's scratch live below 256)
            double mom[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
            for (int i = tid; i < M; i += kRansacThreads)
                if (mask[i]) {
                    const float4 c = pts[i];
                    mom[0] += (double)c.x; mom[1] += (double)c.y; mom[2] += (double)c.z; mom[3] += (double)c.w; mom[4] += 1.0;
                }
            block_tree_sum_many<5>(mom, red_part, red_tot);
            if (!(mom[4] >= (double)Model::kLoMin)) break;
            Norm2d n1, n2;
            const double inv = 1.0 / mom[4];
            n1.cx = mom[0] * inv; n1.cy = mom[1] * inv; n2.cx = mom[2] * inv; n2.cy = mom[3] * inv;
            double dd[2] = {0.0, 0.0};
            for (int i = tid; i < M; i += kRansacThreads)
                if (mask[i]) {
                    const float4 c = pts[i];
                    const double ax = (double)c.x - n1.cx, ay = (double)c.y - n1.cy;
                    const double bx = (double)c.z - n2.cx, by = (double)c.w - n2.cy;
                    dd[0] += sqrt(ax * ax + ay * ay);
                    dd[1] += sqrt(bx * bx + by * by);
                }
            block_tree_sum_many<2>(dd, red_part, red_tot);
            dd[0] *= inv; dd[1] *= inv;
            if (!(dd[0] > 1e-9) || !(dd[1] > 1e-9)) break;
            n1.s = 1.4142135623730951 / dd[0];
            n2.s = 1.4142135623730951 / dd[1];
            double acc[45];
#pragma unroll
            for (int e = 0; e < 45; ++e) acc[e] = 0.0;
            for (int i = tid; i < M; i += kRansacThreads)
                if (mask[i]) {
                    const float4 c = pts[i];
                    const double u1 = ((double)c.x - n1.cx) * n1.s, v1 = ((double)c.y - n1.cy) * n1.s;
                    const double u2 = ((double)c.z - n2.cx) * n2.s, v2 = ((double)c.w - n2.cy) * n2.s;
                    Model::lo_rows(acc, u1, v1, u2, v2);
                }
            double* AtA = S.modelD;              // 81 doubles; the eigen-solver's scratch follows
            block_tree_sum_many<45>(acc, red_part, red_tot);
            if (tid == 0) {
                int e = 0;
                for (int a = 0; a < 9; ++a)
                    for (int b = a; b < 9; ++b) { AtA[a * 9 + b] = acc[e]; AtA[b * 9 + a] = acc[e]; ++e; }
            }
            __syncthreads();
            if (tid == 0) {
                double h[9];
                S.ok = smallest_eigvec9(AtA, S.modelD + 81, h);
                if (S.ok) S.ok = Model::refit(h, n1, n2, S.trialM);
            }
            __syncthreads();
            if (!S.ok) break;
            const int cnt = block_count_inliers<Model>(S.trialM, pts, M, thr2, prm.score, nullptr, &S.total);
            if (cnt <= best) break;
            best = cnt;
            if (tid < 9) S.bestM[tid] = S.trialM[tid];
            __syncthreads();
            block_count_inliers<Model>(S.bestM, pts, M, thr2, prm.score, mask, &S.total);
        }
    }
    __syncthreads();
    if (prm.min_inliers > 0 && best < prm.min_inliers) {
        for (int i = tid; i < M; i += kRansacThreads) mask[i] = 0;
        return;
    }
    if (tid == 0) {
        // cv2 convention model[2,2] == 1.0 exactly: divide (x / x == 1), never multiply by a reciprocal
        const double s = (fabs(S.bestM[8]) > 1.1920928955078125e-07) ? S.bestM[8] : 1.0;
        for (int i = 0; i < 9; ++i) out_model[(long long)p * 9 + i] = S.bestM[i] / s;
        out_ninl[p] = best;
    }
}

// Signature of ransac_f_kernel and ransac_h_kernel (RANSAC-F has no stop target and is launched with a null one)
using RansacKernel = void (*)(const float*, int, const int32_t*, const int32_t*, const uint32_t*, const uint32_t*, const int32_t*,
                              sfm_ransac_params, int, double*, int32_t*, uint8_t*, int32_t*);

// Host side of the four entry points: argument checks, shared-memory sizing and the launch on the caller's current device
template <class Model>
static int launch_ransac(RansacKernel kernel, const float* corr, int corr_stride, const int32_t* count, const int32_t* offsets,
                         int n_pairs, const uint32_t* pair_id, const uint32_t* samples, const int32_t* stop_target,
                         const sfm_ransac_params* prm, double* out_model, int32_t* out_ninl, uint8_t* out_mask, int32_t* out_iters,
                         void* stream)
{
    SFM_REQUIRE(corr && (count || offsets) && prm && out_model && out_ninl && out_mask, "%s: NULL argument", Model::kName);
    if (const int rc = Model::check(*prm)) return rc;
    SFM_REQUIRE(prm->max_iters > 0 && prm->threshold > 0.f, "max_iters and threshold must be positive");
    SFM_REQUIRE(corr_stride > 0 && n_pairs >= 0, "bad sizes");
    SFM_REQUIRE(((uintptr_t)corr & 15) == 0, "corr must be 16-byte aligned");
    if (n_pairs == 0) return SFM_OK;
    const int pts_cap = corr_stride < kPtsCap ? corr_stride : kPtsCap;
    const size_t smem = ransac_smem_fixed<Model>() + (size_t)pts_cap * 16;
    static SmemAttrTable attr;                               // per device and per model
    SFM_CUDA_CHECK(ensure_dyn_smem(kernel, smem, current_device(), attr));
    kernel<<<n_pairs, kRansacThreads, smem, (cudaStream_t)stream>>>(corr, corr_stride, count, offsets, pair_id, samples, stop_target,
                                                                     *prm, pts_cap, out_model, out_ninl, out_mask, out_iters);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return SFM_OK;
}

}  // namespace sfm
