// bundle.cu -- bundle adjustment: registered cameras and triangulated points refined together by Levenberg-Marquardt on the
// Schur-reduced camera system.  Compile with -fmad=false (it shares pose_rows / apply_pose_step with pnp.cu).
//
// include/sfm_b200.h, "bundle adjustment", states the contract.  The call is a fixed launch sequence, so it can be captured
// in a CUDA graph and nothing waits for the host:
//   setup    ba_mark_kernel     one thread per track: used observations, per-image counts, range checks, initial cost
//            ba_setup_kernel    one CTA: the default gauge, camera compaction to 0..Nv-1, list offsets, statuses, state
//            ba_lists_kernel    one CTA per variable camera: its used observations in ascending observation (= track) order
//   per LM iteration (every kernel returns at once after the stop):
//            ba_point_kernel    one thread per track: after an accepted step the per-observation Jacobians, V and the point
//                               gradient; every time the damped V^-1
//            ba_camera_kernel   one CTA per variable camera: U and the gradient (fixed-tree block sums), then its block row of
//                               S = U - W V^-1 W^T and of the reduced gradient, over its observations in ascending track order
//            ba_solve_kernel    cooperative: blocked right-looking Cholesky of S (32 x 32 tiles), the two triangular solves
//                               and the trial camera poses
//            ba_update_kernel   one thread per track: the point back-substitution, the trial cost and the step norms
//            ba_decide_kernel   one CTA: fixed-order totals, accept / reject, lambda by Nielsen's rule, the stop rules
//   output   ba_output_kernel   poses, points, per-observation errors and the summary
// No floating-point atomics: every sum has one owner and a fixed order, so the result is bit-identical run to run.
#include <algorithm>

#include <cooperative_groups.h>

#include "ransac_common.cuh"

namespace cg = cooperative_groups;

namespace sfm {

constexpr int kBaTile = 32;             // Cholesky tile
constexpr int kBaThreads = 256;         // = kRansacThreads: block_tree_sum_many's CTA
constexpr int kBaOne = 1024;            // threads of the single-CTA kernels
constexpr int kBaMaxImages = 1024;
constexpr int kObsTerms = 20;           // per used observation: ju, jv (6 + 6), pu, pv (3 + 3), ex, ey
constexpr int kTrackSums = 4;           // per track: trial cost, |dX|^2, |X|^2, predicted decrease
constexpr double kLambda0 = 1e-4;
constexpr double kLambdaMax = 1e32;

enum BaStatus { kBaFunctionTol = 0, kBaParameterTol = 1, kBaMaxIters = 2, kBaNoProgress = 3, kBaNothing = 4, kBaInvalid = 5, kBaRunning = 6 };

struct BaState {
    int status, nv, npad, cur;          // npad: 6 nv rounded up to the tile; cur: slot (0 / 1) of the current poses and points
    int iters, accepted, relin;         // relin: the next iteration recomputes the Jacobians
    int fail;                           // the trial is rejected: a block not positive definite or a point behind a camera
    int invalid, used_obs, adjusted, pad;
    long long n_tracks, n_obs;
    double lambda, nu, cost, init_cost;
    double cam_pred, cam_dx2, cam_x2;   // the cameras' share of the trial's predicted decrease, |dx|^2 and |x|^2
};

struct BaWork {
    BaState* st;
    int *cidx, *var_img, *img_used, *list_off, *list, *obs_track;
    uint8_t *obs_used, *adjust;
    double *J, *pose, *X, *V, *gp, *Vi, *tsum, *camD, *camG, *rhs, *S;
    size_t bytes;
};

static __host__ __device__ inline long long ba_npad_max(int n_images) { return ((6ll * n_images + kBaTile - 1) / kBaTile) * kBaTile; }

static BaWork carve(void* base, int n_images, long long max_tracks, long long max_obs)
{
    BaWork w{};
    size_t off = 0;
    auto take = [&](size_t bytes) {
        void* p = base ? (void*)((char*)base + off) : nullptr;
        off += (bytes + 255) & ~(size_t)255;
        return p;
    };
    const long long T = std::max(max_tracks, 1ll), O = std::max(max_obs, 1ll), n = n_images, np = ba_npad_max(n_images);
    w.st = (BaState*)take(sizeof(BaState));
    w.cidx = (int*)take(4 * n);
    w.var_img = (int*)take(4 * n);
    w.img_used = (int*)take(4 * n);
    w.list_off = (int*)take(4 * (n + 1));
    w.list = (int*)take(4 * O);
    w.obs_track = (int*)take(4 * O);
    w.obs_used = (uint8_t*)take(O);
    w.adjust = (uint8_t*)take(T);
    w.J = (double*)take(8 * kObsTerms * O);
    w.pose = (double*)take(8 * 2 * 12 * n);
    w.X = (double*)take(8 * 2 * 3 * T);
    w.V = (double*)take(8 * 6 * T);
    w.gp = (double*)take(8 * 3 * T);
    w.Vi = (double*)take(8 * 6 * T);
    w.tsum = (double*)take(8 * kTrackSums * T);
    w.camD = (double*)take(8 * 6 * n);
    w.camG = (double*)take(8 * 6 * n);
    w.rhs = (double*)take(8 * np);
    w.S = (double*)take(8 * np * np);
    w.bytes = off;
    return w;
}

struct BaInputs {
    const int64_t* offsets;
    const int32_t* obs;
    const int64_t* track_counts;
    const uint8_t* point_status;
    const uint8_t* obs_inlier;
    const double* X;
    const float* xy;
    const double* cams;
    const uint8_t* registered;
    const uint8_t* fixed;
    long long max_tracks, max_obs;
    int n_images, S, xy_stride;
};

static __device__ __forceinline__ bool ba_finite(double v) { return fabs(v) <= 1.7976931348623157e308; }

static __device__ __forceinline__ void ba_normalised(const BaInputs& in, int img, int f, double& x, double& y)
{
    const float* p = in.xy + 2 * ((long long)img * in.xy_stride + f);
    const double* c = in.cams + 16ll * img;
    x = ((double)__ldg(p) - __ldg(c + 2)) / __ldg(c + 0);
    y = ((double)__ldg(p + 1) - __ldg(c + 3)) / __ldg(c + 1);
}

// Camera img of pose slot s: intrinsics from the table, R and t from the slot
static __device__ __forceinline__ void ba_camera(const BaInputs& in, const BaWork& w, int s, int img, Camera& K)
{
    K.fx = __ldg(in.cams + 16ll * img);
    K.fy = __ldg(in.cams + 16ll * img + 1);
    const double* p = w.pose + (12ll * in.n_images) * s + 12ll * img;
#pragma unroll
    for (int i = 0; i < 9; ++i) K.r[i] = p[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) K.t[i] = p[9 + i];
}

// Squared pixel residual without the cheirality test (the cost counts every used observation)
static __device__ __forceinline__ double ba_sq(const Camera& K, const double* X, double x, double y, double& p2)
{
    const double p0 = K.r[0] * X[0] + K.r[1] * X[1] + K.r[2] * X[2] + K.t[0];
    const double p1 = K.r[3] * X[0] + K.r[4] * X[1] + K.r[5] * X[2] + K.t[1];
    p2 = K.r[6] * X[0] + K.r[7] * X[1] + K.r[8] * X[2] + K.t[2];
    const double iz = 1.0 / p2;
    const double ex = (p0 * iz - x) * K.fx;
    const double ey = (p1 * iz - y) * K.fy;
    return ex * ex + ey * ey;
}

static __device__ __forceinline__ long long ba_tracks(const BaInputs& in) { return min((long long)__ldg(in.track_counts), in.max_tracks); }

// Fixed-order sum over the 1,024 threads of a single-CTA kernel: shuffle trees per warp, then the 32 warp sums in order
template <int N>
static __device__ __forceinline__ void ba_block_sum(double (&v)[N], double* part)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int e = 0; e < N; ++e) {
        double x = v[e];
        for (int off = 16; off >= 1; off >>= 1) x += __shfl_down_sync(0xffffffffu, x, off);
        if (lane == 0) part[e * 32 + warp] = x;
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < N; ++e) {
        double t = part[e * 32];
        for (int i = 1; i < 32; ++i) t += part[e * 32 + i];
        v[e] = t;
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------------------ setup
__global__ void __launch_bounds__(kBaThreads) ba_mark_kernel(BaInputs in, BaWork w)
{
    const long long n_tracks = ba_tracks(in);
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < in.max_tracks; k += (long long)gridDim.x * blockDim.x) {
        double X[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            X[c] = __ldg(in.X + 3 * k + c);
            w.X[3 * k + c] = X[c];
            w.X[3 * in.max_tracks + 3 * k + c] = X[c];
        }
        if (k >= n_tracks) continue;
        const long long o0 = min((long long)__ldg(in.offsets + k), in.max_obs), o1 = min((long long)__ldg(in.offsets + k + 1), in.max_obs);
        const bool has_point = __ldg(in.point_status + k) == 0;
        int n_used = 0;
        bool bad = false;
        double cost = 0.0;
        for (long long o = o0; o < o1; ++o) {
            const int img = __ldg(in.obs + 2 * o), f = __ldg(in.obs + 2 * o + 1);
            const bool in_range = img >= 0 && img < in.n_images && f >= 0 && f < in.S;
            bad |= has_point && !in_range;
            const bool used = has_point && in_range && __ldg(in.obs_inlier + o) == 1 && (!in.registered || __ldg(in.registered + img));
            w.obs_track[o] = (int)k;
            w.obs_used[o] = (uint8_t)used;
            if (used) {
                ++n_used;
                atomicAdd(w.img_used + img, 1);
                double x, y, p2;
                ba_normalised(in, img, f, x, y);
                Camera K;
                load_camera(in.cams + 16ll * img, K);
                cost = cost + ba_sq(K, X, x, y, p2);
            }
        }
        w.adjust[k] = (uint8_t)(n_used >= 2);
        w.tsum[kTrackSums * k] = cost;
        if (bad) atomicOr(&w.st->invalid, 1);
        if (n_used) atomicAdd(&w.st->used_obs, n_used);
        if (n_used >= 2) atomicAdd(&w.st->adjusted, 1);
    }
}

__global__ void __launch_bounds__(kBaOne) ba_setup_kernel(BaInputs in, BaWork w)
{
    __shared__ int scan_v[kBaOne], scan_u[kBaOne];
    __shared__ int gauge, bad_focal;
    __shared__ double part[32];
    const int i = threadIdx.x;
    if (i == 0) { gauge = kBaOne; bad_focal = 0; }
    __syncthreads();
    const bool reg = i < in.n_images && (!in.registered || in.registered[i]);
    if (!in.fixed && reg) atomicMin(&gauge, i);
    const int used = i < in.n_images ? w.img_used[i] : 0;
    if (i < in.n_images && reg && used > 0) {
        const double fx = __ldg(in.cams + 16ll * i), fy = __ldg(in.cams + 16ll * i + 1);
        if (!(fx > 0.0) || !(fy > 0.0) || !ba_finite(fx) || !ba_finite(fy)) atomicOr(&bad_focal, 1);
    }
    if (i < in.n_images)
        for (int e = 0; e < 12; ++e) {
            const double v = __ldg(in.cams + 16ll * i + 4 + e);
            w.pose[12 * i + e] = v;
            w.pose[12ll * in.n_images + 12 * i + e] = v;
        }
    __syncthreads();
    const bool fixed = in.fixed ? (i < in.n_images && in.fixed[i] != 0) : i == gauge;
    const int var = reg && !fixed && used > 0;
    scan_v[i] = var;
    scan_u[i] = var ? used : 0;
    __syncthreads();
    for (int d = 1; d < kBaOne; d <<= 1) {          // inclusive Hillis-Steele scans (integers: exact)
        const int a = i >= d ? scan_v[i - d] : 0, b = i >= d ? scan_u[i - d] : 0;
        __syncthreads();
        scan_v[i] += a;
        scan_u[i] += b;
        __syncthreads();
    }
    if (i < in.n_images) {
        w.cidx[i] = var ? scan_v[i] - 1 : -1;
        if (var) w.var_img[scan_v[i] - 1] = i;
        w.list_off[i] = scan_u[i] - (var ? used : 0);
        if (i == in.n_images - 1) w.list_off[in.n_images] = scan_u[i];
    }
    // the initial cost: tracks k = i, i + 1024, ... per thread, then the fixed tree (depends only on the track count)
    const long long n_tracks = ba_tracks(in);
    double c[1] = {0.0};
    for (long long k = i; k < n_tracks; k += kBaOne) c[0] = c[0] + w.tsum[kTrackSums * k];
    ba_block_sum<1>(c, part);
    if (i == 0) {
        BaState& s = *w.st;
        s.nv = scan_v[kBaOne - 1];
        s.npad = (int)(((6ll * s.nv + kBaTile - 1) / kBaTile) * kBaTile);
        s.cur = 0; s.iters = 0; s.accepted = 0; s.relin = 1; s.fail = 0;
        s.n_tracks = n_tracks;
        s.n_obs = n_tracks > 0 ? min((long long)__ldg(in.offsets + n_tracks), in.max_obs) : 0;
        s.lambda = kLambda0; s.nu = 2.0;
        s.cost = c[0]; s.init_cost = c[0];
        if (s.invalid || bad_focal) s.status = kBaInvalid;
        else if (s.nv == 0 && s.adjusted == 0) s.status = kBaNothing;
        else s.status = kBaRunning;
    }
}

// The used observations of variable camera blockIdx.x, in ascending observation index (tracks list theirs in track order)
__global__ void __launch_bounds__(kBaThreads) ba_lists_kernel(BaInputs in, BaWork w)
{
    __shared__ int warp_total[kBaThreads / 32];
    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (w.st->status != kBaRunning || w.cidx[img] < 0) return;
    const long long n_obs = w.st->n_obs;
    int base = w.list_off[img];
    for (long long o0 = 0; o0 < n_obs; o0 += kBaThreads) {
        const long long o = o0 + tid;
        const bool use = o < n_obs && w.obs_used[o] && __ldg(in.obs + 2 * o) == img;
        const unsigned bal = __ballot_sync(0xffffffffu, use);
        if (lane == 0) warp_total[warp] = __popc(bal);
        __syncthreads();
        int off = base, total = 0;
#pragma unroll
        for (int v = 0; v < kBaThreads / 32; ++v) {
            off += v < warp ? warp_total[v] : 0;
            total += warp_total[v];
        }
        if (use) w.list[off + __popc(bal & ((1u << lane) - 1u))] = (int)o;
        base += total;
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------------ iteration
__global__ void __launch_bounds__(kBaThreads) ba_point_kernel(BaInputs in, BaWork w)
{
    const BaState& s = *w.st;
    if (s.status != kBaRunning) return;
    const int cur = s.cur, relin = s.relin;
    const double lambda = s.lambda;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < s.n_tracks; k += (long long)gridDim.x * blockDim.x) {
        const bool adj = w.adjust[k];
        if (relin) {
            const long long o0 = min((long long)__ldg(in.offsets + k), in.max_obs), o1 = min((long long)__ldg(in.offsets + k + 1), in.max_obs);
            const double* X = w.X + 3 * in.max_tracks * cur + 3 * k;
            const double Xk[3] = {X[0], X[1], X[2]};
            double v[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};     // V (00 01 02 11 12 22), then the point gradient
            for (long long o = o0; o < o1; ++o) {
                if (!w.obs_used[o]) continue;
                const int img = __ldg(in.obs + 2 * o);
                double x, y;
                ba_normalised(in, img, __ldg(in.obs + 2 * o + 1), x, y);
                Camera K;
                ba_camera(in, w, cur, img, K);
                PoseRows P;
                pose_rows(K, x, y, Xk, P);
                double pu[3], pv[3];
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    pu[c] = P.a0 * K.r[c] + P.a2 * K.r[6 + c];
                    pv[c] = P.b1 * K.r[3 + c] + P.b2 * K.r[6 + c];
                }
                double* J = w.J + kObsTerms * o;
#pragma unroll
                for (int c = 0; c < 6; ++c) { J[c] = P.ju[c]; J[6 + c] = P.jv[c]; }
#pragma unroll
                for (int c = 0; c < 3; ++c) { J[12 + c] = pu[c]; J[15 + c] = pv[c]; }
                J[18] = P.ex; J[19] = P.ey;
                int e = 0;
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int b = a; b < 3; ++b) {
                        v[e] = v[e] + pu[a] * pu[b];
                        v[e] = v[e] + pv[a] * pv[b];
                        ++e;
                    }
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    v[6 + a] = v[6 + a] + pu[a] * P.ex;
                    v[6 + a] = v[6 + a] + pv[a] * P.ey;
                }
            }
            if (adj) {
#pragma unroll
                for (int e = 0; e < 6; ++e) w.V[6 * k + e] = v[e];
#pragma unroll
                for (int e = 0; e < 3; ++e) w.gp[3 * k + e] = v[6 + e];
            }
        }
        if (!adj) continue;
        const double* V = w.V + 6 * k;
        const double d00 = V[0] + lambda * V[0], d01 = V[1], d02 = V[2], d11 = V[3] + lambda * V[3], d12 = V[4], d22 = V[5] + lambda * V[5];
        const double c00 = d11 * d22 - d12 * d12, c01 = d02 * d12 - d01 * d22, c02 = d01 * d12 - d02 * d11;
        const double c11 = d00 * d22 - d02 * d02, c12 = d01 * d02 - d00 * d12, c22 = d00 * d11 - d01 * d01;
        const double det = d00 * c00 + d01 * c01 + d02 * c02;
        if (!(det > 0.0) || !ba_finite(det)) atomicOr(&w.st->fail, 1);
        const double id = 1.0 / det;
        double* Vi = w.Vi + 6 * k;
        Vi[0] = c00 * id; Vi[1] = c01 * id; Vi[2] = c02 * id; Vi[3] = c11 * id; Vi[4] = c12 * id; Vi[5] = c22 * id;
    }
}

static __device__ __forceinline__ void sym3_mul(const double* M, const double* x, double* y)
{
    y[0] = M[0] * x[0] + M[1] * x[1] + M[2] * x[2];
    y[1] = M[1] * x[0] + M[3] * x[1] + M[4] * x[2];
    y[2] = M[2] * x[0] + M[4] * x[1] + M[5] * x[2];
}

// Block row a of S (columns of cameras b <= a) and of the reduced right-hand side -g_a + sum W V^-1 g_p.  The observations of
// camera a are visited one at a time in ascending track order; within one, the threads take the track's other observations
// (a run of observations of one image has one owner: tracks list observations by ascending node), so every block entry is
// updated by one thread at a time, in track order.
__global__ void __launch_bounds__(kBaThreads) ba_camera_kernel(BaInputs in, BaWork w)
{
    __shared__ double part[27 * 8], tot[27];
    const BaState& s = *w.st;
    const int img = blockIdx.x, tid = threadIdx.x;
    if (s.status != kBaRunning || s.fail || w.cidx[img] < 0) return;
    const int a = w.cidx[img], ld = s.npad;
    const double lambda = s.lambda;
    const int l0 = w.list_off[img], l1 = w.list_off[img + 1];
    double v[27];
#pragma unroll
    for (int e = 0; e < 27; ++e) v[e] = 0.0;
    for (int e = l0 + tid; e < l1; e += kBaThreads) {
        const double* J = w.J + kObsTerms * (long long)w.list[e];
        double ju[6], jv[6];
#pragma unroll
        for (int c = 0; c < 6; ++c) { ju[c] = J[c]; jv[c] = J[6 + c]; }
        int q = 0;
#pragma unroll
        for (int i = 0; i < 6; ++i)
#pragma unroll
            for (int j = i; j < 6; ++j) {
                v[q] = v[q] + ju[i] * ju[j];
                v[q] = v[q] + jv[i] * jv[j];
                ++q;
            }
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            v[21 + i] = v[21 + i] + ju[i] * J[18];
            v[21 + i] = v[21 + i] + jv[i] * J[19];
        }
    }
    block_tree_sum_many<27>(v, part, tot);
    double* row = w.S + (long long)(6 * a) * ld;
    for (int e = tid; e < 6 * (6 * a + 6); e += kBaThreads) {
        const int r = e / (6 * a + 6), c = e - r * (6 * a + 6);
        double val = 0.0;
        if (c >= 6 * a) {
            const int i = min(r, c - 6 * a), j = max(r, c - 6 * a);
            val = tot[i * 6 - i * (i - 1) / 2 + (j - i)];      // (shared: indexed at run time)
            if (i == j) val = val + lambda * val;
        }
        row[(long long)r * ld + c] = val;
    }
    if (tid < 6) {
        w.camD[6 * a + tid] = tot[tid * 6 - tid * (tid - 1) / 2];
        w.camG[6 * a + tid] = tot[21 + tid];
    }
    double rg[6] = {0, 0, 0, 0, 0, 0};
    __syncthreads();
    for (int e = l0; e < l1; ++e) {
        const long long o = w.list[e];
        const long long k = w.obs_track[o];
        if (!w.adjust[k]) continue;                  // a point held fixed adds no Schur term
        const double* J = w.J + kObsTerms * o;
        const double* Vi = w.Vi + 6 * k;
        double su[3], sv[3];
        sym3_mul(Vi, J + 12, su);                    // V^-1 pu, V^-1 pv: W_o V^-1 = ju su^T + jv sv^T
        sym3_mul(Vi, J + 15, sv);
        if (tid == 0) {
            const double* g = w.gp + 3 * k;
            const double au = su[0] * g[0] + su[1] * g[1] + su[2] * g[2];
            const double av = sv[0] * g[0] + sv[1] * g[1] + sv[2] * g[2];
#pragma unroll
            for (int r = 0; r < 6; ++r) rg[r] = rg[r] + (J[r] * au + J[6 + r] * av);
        }
        const long long t0 = min((long long)__ldg(in.offsets + k), in.max_obs), t1 = min((long long)__ldg(in.offsets + k + 1), in.max_obs);
        for (long long j = t0 + tid; j < t1; j += kBaThreads) {
            const int ij = __ldg(in.obs + 2 * j);
            if (j > t0 && __ldg(in.obs + 2 * (j - 1)) == ij) continue;       // not the first of its image's run
            if (ij < 0 || ij >= in.n_images) continue;
            const int b = w.cidx[ij];
            if (b < 0 || b > a) continue;
            double* blk = row + 6 * b;
            for (long long jj = j; jj < t1 && __ldg(in.obs + 2 * jj) == ij; ++jj) {
                if (!w.obs_used[jj]) continue;
                const double* Q = w.J + kObsTerms * jj;
                const double al = su[0] * Q[12] + su[1] * Q[13] + su[2] * Q[14];
                const double be = su[0] * Q[15] + su[1] * Q[16] + su[2] * Q[17];
                const double ga = sv[0] * Q[12] + sv[1] * Q[13] + sv[2] * Q[14];
                const double de = sv[0] * Q[15] + sv[1] * Q[16] + sv[2] * Q[17];
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                    const double mu = al * Q[c] + be * Q[6 + c], mv = ga * Q[c] + de * Q[6 + c];
#pragma unroll
                    for (int r = 0; r < 6; ++r) blk[(long long)r * ld + c] = blk[(long long)r * ld + c] - (J[r] * mu + J[6 + r] * mv);
                }
            }
        }
        __syncthreads();
    }
    if (tid == 0)
        for (int r = 0; r < 6; ++r) w.rhs[6 * a + r] = rg[r] - v[21 + r];
}

// ------------------------------------------------------------------------------------------------------------ factor + solve
struct CholSmem {
    double A[kBaTile][kBaTile + 1];
    double B[kBaTile][kBaTile + 1];
};

static __device__ __forceinline__ bool ba_failed(const BaState* st) { return *(volatile const int*)&st->fail != 0; }

// The lower-triangular tile pair index t -> (i, j), j <= i
static __device__ __forceinline__ void tri_index(long long t, int& i, int& j)
{
    int r = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
    while ((long long)r * (r + 1) / 2 > t) --r;
    while ((long long)(r + 1) * (r + 2) / 2 <= t) ++r;
    i = r;
    j = (int)(t - (long long)r * (r + 1) / 2);
}

// The lower triangle of diagonal tile k0 into sm.A (the upper part is zero); the caller's CTA only
static __device__ __forceinline__ void diag_tile_to_smem(const double* S, long long ld, long long k0, CholSmem& sm)
{
    __syncthreads();
    for (int e = threadIdx.x; e < kBaTile * kBaTile; e += kBaThreads) {
        const int r = e / kBaTile, c = e % kBaTile;
        sm.A[r][c] = c <= r ? S[(k0 + r) * ld + k0 + c] : 0.0;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kBaThreads) ba_solve_kernel(BaInputs in, BaWork w)
{
    __shared__ CholSmem sm;
    cg::grid_group grid = cg::this_grid();
    BaState* st = w.st;
    if (st->status != kBaRunning || st->fail) return;            // uniform over the grid: nothing below changes them first
    const int tid = threadIdx.x, nv = st->nv, N = st->npad, nb = N / kBaTile, cur = st->cur;
    const long long ld = N;
    double* S = w.S;
    double* y = w.rhs;
    const long long gt = (long long)blockIdx.x * kBaThreads + tid, gn = (long long)gridDim.x * kBaThreads;
    // padding rows past 6 nv: the identity, right-hand side 0
    for (long long e = gt; e < (long long)(N - 6 * nv) * N; e += gn) {
        const long long r = 6 * nv + e / N, c = e % N;
        if (c <= r) S[r * ld + c] = c == r ? 1.0 : 0.0;
        if (c == 0) y[r] = 0.0;
    }
    grid.sync();
    bool ok = true;
    for (int kb = 0; kb < nb && ok; ++kb) {
        const long long k0 = (long long)kb * kBaTile;
        if (blockIdx.x == 0) {                                  // the diagonal tile
            for (int e = tid; e < kBaTile * kBaTile; e += kBaThreads) sm.A[e / kBaTile][e % kBaTile] = S[(k0 + e / kBaTile) * ld + k0 + e % kBaTile];
            __syncthreads();
            for (int j = 0; j < kBaTile; ++j) {
                if (tid == 0) {
                    const double d = sm.A[j][j];
                    if (!(d > 0.0) || !ba_finite(d)) st->fail = 1;
                    sm.A[j][j] = sqrt(d);
                }
                __syncthreads();
                if (tid > j && tid < kBaTile) sm.A[tid][j] = sm.A[tid][j] / sm.A[j][j];
                __syncthreads();
                for (int e = tid; e < kBaTile * kBaTile; e += kBaThreads) {
                    const int r = e / kBaTile, c = e % kBaTile;
                    if (c > j && r >= c) sm.A[r][c] = sm.A[r][c] - sm.A[r][j] * sm.A[c][j];
                }
                __syncthreads();
            }
            for (int e = tid; e < kBaTile * kBaTile; e += kBaThreads) {
                const int r = e / kBaTile, c = e % kBaTile;
                if (c <= r) S[(k0 + r) * ld + k0 + c] = sm.A[r][c];
            }
        }
        grid.sync();
        if (ba_failed(st)) { ok = false; break; }
        // the panel: L_ik = A_ik L_kk^-T, one CTA per tile, column by column in shared memory
        diag_tile_to_smem(S, ld, k0, sm);
        for (int i = kb + 1 + blockIdx.x; i < nb; i += gridDim.x) {
            double* tile = S + (long long)i * kBaTile * ld + k0;
            __syncthreads();
            for (int e = tid; e < kBaTile * kBaTile; e += kBaThreads) sm.B[e / kBaTile][e % kBaTile] = tile[(e / kBaTile) * ld + e % kBaTile];
            __syncthreads();
            for (int c = 0; c < kBaTile; ++c) {
                if (tid < kBaTile) sm.B[tid][c] = sm.B[tid][c] / sm.A[c][c];
                __syncthreads();
                for (int e = tid; e < kBaTile * kBaTile; e += kBaThreads) {
                    const int r = e / kBaTile, cc = e % kBaTile;
                    if (cc > c) sm.B[r][cc] = sm.B[r][cc] - sm.B[r][c] * sm.A[cc][c];
                }
                __syncthreads();
            }
            for (int e = tid; e < kBaTile * kBaTile; e += kBaThreads) tile[(e / kBaTile) * ld + e % kBaTile] = sm.B[e / kBaTile][e % kBaTile];
        }
        grid.sync();
        // the trailing update: A_ij -= L_ik L_jk^T for kb < j <= i
        const int m = nb - kb - 1;
        const long long n_tiles = (long long)m * (m + 1) / 2;
        for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            int ii, jj;
            tri_index(t, ii, jj);
            const long long i0 = (long long)(kb + 1 + ii) * kBaTile, j0 = (long long)(kb + 1 + jj) * kBaTile;
            __syncthreads();
            for (int e = tid; e < kBaTile * kBaTile; e += kBaThreads) {
                const int r = e / kBaTile, c = e % kBaTile;
                sm.A[r][c] = S[(i0 + r) * ld + k0 + c];
                sm.B[r][c] = S[(j0 + r) * ld + k0 + c];
            }
            __syncthreads();
            const int r = tid >> 3;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int c = (tid & 7) + 8 * q;
                double acc = 0.0;
#pragma unroll
                for (int mm = 0; mm < kBaTile; ++mm) acc = acc + sm.A[r][mm] * sm.B[c][mm];
                double* p = S + (i0 + r) * ld + j0 + c;
                *p = *p - acc;
            }
        }
        grid.sync();
    }
    if (!ok) return;                                            // every CTA saw the same flag after the same barrier
    // L z = rhs, then L^T dc = z: a tile's unknowns by one warp (lane = row, column by column), the other rows' updates
    // spread over the grid
    for (int kb = 0; kb < nb; ++kb) {
        const long long k0 = (long long)kb * kBaTile;
        if (blockIdx.x == 0) {
            diag_tile_to_smem(S, ld, k0, sm);
            if (tid < 32) {
                double b = y[k0 + tid];
                for (int c = 0; c < kBaTile; ++c) {
                    if (tid == c) b = b / sm.A[c][c];
                    const double yc = __shfl_sync(0xffffffffu, b, c);
                    if (tid > c) b = b - sm.A[tid][c] * yc;
                }
                y[k0 + tid] = b;
            }
        }
        grid.sync();
        for (long long r = k0 + kBaTile + gt; r < N; r += gn) {
            double acc = 0.0;
            for (int mm = 0; mm < kBaTile; ++mm) acc = acc + S[r * ld + k0 + mm] * y[k0 + mm];
            y[r] = y[r] - acc;
        }
        grid.sync();
    }
    for (int kb = nb - 1; kb >= 0; --kb) {
        const long long k0 = (long long)kb * kBaTile;
        if (blockIdx.x == 0) {
            diag_tile_to_smem(S, ld, k0, sm);
            if (tid < 32) {
                double b = y[k0 + tid];
                for (int c = kBaTile - 1; c >= 0; --c) {
                    if (tid == c) b = b / sm.A[c][c];
                    const double xc = __shfl_sync(0xffffffffu, b, c);
                    if (tid < c) b = b - sm.A[c][tid] * xc;
                }
                y[k0 + tid] = b;
            }
        }
        grid.sync();
        for (long long r = gt; r < k0; r += gn) {
            double acc = 0.0;
            for (int mm = 0; mm < kBaTile; ++mm) acc = acc + S[(k0 + mm) * ld + r] * y[k0 + mm];
            y[r] = y[r] - acc;
        }
        grid.sync();
    }
    // the trial poses of the variable cameras, and the cameras' share of the step statistics
    for (long long a = gt; a < nv; a += gn) {
        const int img = w.var_img[a];
        Camera K, O;
        ba_camera(in, w, cur, img, K);
        apply_pose_step(y + 6 * a, K, O);
        double* p = w.pose + (12ll * in.n_images) * (1 - cur) + 12ll * img;
#pragma unroll
        for (int i = 0; i < 9; ++i) p[i] = O.r[i];
#pragma unroll
        for (int i = 0; i < 3; ++i) p[9 + i] = O.t[i];
    }
    if (blockIdx.x == 0 && tid == 0) {
        const double lambda = st->lambda;
        double pred = 0.0, dx2 = 0.0, x2 = 0.0;
        for (int a = 0; a < nv; ++a) {
            const double* t = w.pose + (12ll * in.n_images) * cur + 12ll * w.var_img[a] + 9;
            for (int r = 0; r < 6; ++r) {
                const double h = y[6 * a + r];
                pred = pred + h * (lambda * w.camD[6 * a + r] * h - w.camG[6 * a + r]);
                dx2 = dx2 + h * h;
            }
            x2 = x2 + (t[0] * t[0] + t[1] * t[1] + t[2] * t[2]);
        }
        st->cam_pred = pred; st->cam_dx2 = dx2; st->cam_x2 = x2;
    }
}

// ------------------------------------------------------------------------------------------------------------ update + decide
__global__ void __launch_bounds__(kBaThreads) ba_update_kernel(BaInputs in, BaWork w)
{
    const BaState& s = *w.st;
    if (s.status != kBaRunning || s.fail) return;
    const int cur = s.cur, nxt = 1 - cur;
    const double lambda = s.lambda;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < s.n_tracks; k += (long long)gridDim.x * blockDim.x) {
        const long long o0 = min((long long)__ldg(in.offsets + k), in.max_obs), o1 = min((long long)__ldg(in.offsets + k + 1), in.max_obs);
        const bool adj = w.adjust[k];
        const double* Xc = w.X + 3 * in.max_tracks * cur + 3 * k;
        double X[3] = {Xc[0], Xc[1], Xc[2]};
        double sums[kTrackSums] = {0.0, 0.0, 0.0, 0.0};
        if (adj) {
            const double* g = w.gp + 3 * k;
            double r[3] = {-g[0], -g[1], -g[2]};
            for (long long o = o0; o < o1; ++o) {
                if (!w.obs_used[o]) continue;
                const int b = w.cidx[__ldg(in.obs + 2 * o)];
                if (b < 0) continue;
                const double* J = w.J + kObsTerms * o;
                const double* h = w.rhs + 6 * b;
                double du = 0.0, dv = 0.0;
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                    du = du + J[c] * h[c];
                    dv = dv + J[6 + c] * h[c];
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) r[c] = r[c] - (J[12 + c] * du + J[15 + c] * dv);
            }
            double dX[3];
            sym3_mul(w.Vi + 6 * k, r, dX);
            const double* V = w.V + 6 * k;
            const double Vd[3] = {V[0], V[3], V[5]};
            double* Xn = w.X + 3 * in.max_tracks * nxt + 3 * k;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                sums[1] = sums[1] + dX[c] * dX[c];
                sums[2] = sums[2] + X[c] * X[c];
                sums[3] = sums[3] + dX[c] * (lambda * Vd[c] * dX[c] - g[c]);
                X[c] = X[c] + dX[c];
                Xn[c] = X[c];
            }
        }
        bool behind = false;
        for (long long o = o0; o < o1; ++o) {
            if (!w.obs_used[o]) continue;
            const int img = __ldg(in.obs + 2 * o);
            double x, y, p2;
            ba_normalised(in, img, __ldg(in.obs + 2 * o + 1), x, y);
            Camera K;
            ba_camera(in, w, nxt, img, K);
            sums[0] = sums[0] + ba_sq(K, X, x, y, p2);
            behind |= !(p2 > 0.0);
        }
        if (behind) atomicOr(&w.st->fail, 1);
#pragma unroll
        for (int e = 0; e < kTrackSums; ++e) w.tsum[kTrackSums * k + e] = sums[e];
    }
}

__global__ void __launch_bounds__(kBaOne) ba_decide_kernel(int max_iters, double ftol, double ptol, BaWork w)
{
    __shared__ double part[kTrackSums * 32];
    BaState& s = *w.st;
    if (s.status != kBaRunning) return;
    const bool failed = s.fail != 0;
    double v[kTrackSums] = {0.0, 0.0, 0.0, 0.0};
    if (!failed) {
        for (long long k = threadIdx.x; k < s.n_tracks; k += kBaOne)
#pragma unroll
            for (int e = 0; e < kTrackSums; ++e) v[e] = v[e] + w.tsum[kTrackSums * k + e];
        ba_block_sum<kTrackSums>(v, part);
    }
    if (threadIdx.x != 0) return;
    const double new_cost = v[0];
    const double pred = s.cam_pred + v[3];
    const double dx = sqrt(s.cam_dx2 + v[1]), xn = sqrt(s.cam_x2 + v[2]);
    s.iters += 1;
    if (!failed && ba_finite(new_cost) && pred > 0.0 && new_cost < s.cost) {
        const double rho = (s.cost - new_cost) / pred;
        const double q = 2.0 * rho - 1.0;
        s.lambda = s.lambda * fmax(1.0 / 3.0, 1.0 - q * q * q);
        s.nu = 2.0;
        const double old = s.cost;
        s.cost = new_cost;
        s.cur = 1 - s.cur;
        s.accepted += 1;
        s.relin = 1;
        if (old - new_cost < ftol * old) s.status = kBaFunctionTol;
        else if (dx <= ptol * (xn + ptol)) s.status = kBaParameterTol;
    } else {
        s.lambda = s.lambda * s.nu;
        s.nu = s.nu * 2.0;
        s.relin = 0;
        if (!(s.lambda <= kLambdaMax)) s.status = kBaNoProgress;
    }
    s.fail = 0;
    if (s.status == kBaRunning && s.iters >= max_iters) s.status = kBaMaxIters;
}

// ------------------------------------------------------------------------------------------------------------ output
__global__ void __launch_bounds__(kBaThreads) ba_output_kernel(BaInputs in, BaWork w, double* __restrict__ out_pose, double* __restrict__ out_X,
                                                               float* __restrict__ out_obs_error, sfm_bundle_summary* __restrict__ out_summary)
{
    const BaState& s = *w.st;
    const int cur = s.cur;
    const long long gt = (long long)blockIdx.x * blockDim.x + threadIdx.x, gn = (long long)gridDim.x * blockDim.x;
    for (long long e = gt; e < 12ll * in.n_images; e += gn) out_pose[e] = w.pose[(12ll * in.n_images) * cur + e];
    for (long long e = gt; e < 3 * in.max_tracks; e += gn) {
        const long long k = e / 3;
        out_X[e] = (k < s.n_tracks && w.adjust[k]) ? w.X[3 * in.max_tracks * cur + e] : __ldg(in.X + e);
    }
    for (long long o = gt; o < s.n_obs; o += gn) {
        float err = __int_as_float(0x7fc00000);
        const long long k = w.obs_track[o];
        const int img = __ldg(in.obs + 2 * o), f = __ldg(in.obs + 2 * o + 1);
        if (__ldg(in.point_status + k) == 0 && img >= 0 && img < in.n_images && f >= 0 && f < in.S &&
            (!in.registered || __ldg(in.registered + img))) {
            double x, y, e2;
            ba_normalised(in, img, f, x, y);
            Camera K;
            ba_camera(in, w, cur, img, K);
            const double* Xk = w.adjust[k] ? w.X + 3 * in.max_tracks * cur + 3 * k : in.X + 3 * k;
            reproject(K, Xk, x, y, 0.0, e2);
            err = (float)sqrt(e2);
        }
        out_obs_error[o] = err;
    }
    if (gt == 0) {
        sfm_bundle_summary r;
        r.status = s.status == kBaRunning ? kBaMaxIters : s.status;
        r.iterations = s.iters;
        r.accepted = s.accepted;
        r.used_obs = s.used_obs;
        r.variable_cameras = s.nv;
        r.adjusted_points = s.adjusted;
        r.initial_cost = s.init_cost;
        r.final_cost = s.cost;
        *out_summary = r;
    }
}

static unsigned ba_grid(long long work, int sms)
{
    return (unsigned)std::max(1ll, std::min((work + kBaThreads - 1) / kBaThreads, 16ll * sms));
}

}  // namespace sfm

using namespace sfm;

extern "C" int sfm_bundle_workspace_bytes(int n_images, int64_t max_tracks, int64_t max_obs, size_t* out_bytes)
{
    SFM_REQUIRE(out_bytes, "sfm_bundle_workspace_bytes: NULL argument");
    SFM_REQUIRE(n_images > 0 && n_images <= kBaMaxImages, "sfm_bundle_workspace_bytes: n_images must lie in [1, %d], got %d", kBaMaxImages,
                n_images);
    SFM_REQUIRE(max_tracks >= 0 && max_obs >= 0 && max_obs < (1ll << 31) && max_tracks < (1ll << 31),
                "sfm_bundle_workspace_bytes: max_tracks and max_obs must lie in [0, 2^31)");
    *out_bytes = carve(nullptr, n_images, max_tracks, max_obs).bytes;
    return SFM_OK;
}

extern "C" int sfm_bundle_adjust(int n_images, int S, const int64_t* offsets, const int32_t* obs, const int64_t* track_counts,
                                 int64_t max_tracks, int64_t max_obs, const uint8_t* point_status, const uint8_t* obs_inlier, const double* X,
                                 const float* xy, int xy_stride, const double* cams, const uint8_t* registered, const uint8_t* fixed,
                                 const sfm_bundle_params* params, void* workspace, size_t workspace_bytes, double* out_pose, double* out_X,
                                 float* out_obs_error, sfm_bundle_summary* out_summary, void* stream)
{
    SFM_REQUIRE(params, "sfm_bundle_adjust: NULL params");
    SFM_REQUIRE(offsets && obs && track_counts && point_status && obs_inlier && X && xy && cams && workspace && out_pose && out_X &&
                    out_obs_error && out_summary,
                "sfm_bundle_adjust: NULL argument");
    SFM_REQUIRE(n_images > 0 && n_images <= kBaMaxImages, "sfm_bundle_adjust: n_images must lie in [1, %d], got %d", kBaMaxImages, n_images);
    SFM_REQUIRE(S > 0, "sfm_bundle_adjust: S must be positive");
    SFM_REQUIRE((long long)n_images * S < (1ll << 31), "sfm_bundle_adjust: n_images * S = %lld must stay below 2^31", (long long)n_images * S);
    SFM_REQUIRE(xy_stride >= S, "sfm_bundle_adjust: xy_stride %d is below S = %d", xy_stride, S);
    SFM_REQUIRE(max_tracks >= 0 && max_obs >= 0 && max_obs < (1ll << 31) && max_tracks < (1ll << 31),
                "sfm_bundle_adjust: max_tracks and max_obs must lie in [0, 2^31)");
    SFM_REQUIRE(params->max_iters >= 1 && params->max_iters <= 10000, "sfm_bundle_adjust: max_iters must lie in [1, 10000], got %d",
                params->max_iters);
    SFM_REQUIRE(params->function_tolerance >= 0.0 && params->function_tolerance < 1e300,
                "sfm_bundle_adjust: function_tolerance must be non-negative and finite, got %g", params->function_tolerance);
    SFM_REQUIRE(params->parameter_tolerance >= 0.0 && params->parameter_tolerance < 1e300,
                "sfm_bundle_adjust: parameter_tolerance must be non-negative and finite, got %g", params->parameter_tolerance);
    const BaWork w = carve(workspace, n_images, max_tracks, max_obs);
    SFM_REQUIRE(workspace_bytes >= w.bytes, "sfm_bundle_adjust: workspace of %zu bytes, %zu needed", workspace_bytes, w.bytes);
    SFM_REQUIRE(((uintptr_t)workspace & 255) == 0, "sfm_bundle_adjust: workspace must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int dev = current_device();
    int sms = 0, coop = 0, per_sm = 0;
    SFM_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    SFM_CUDA_CHECK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    SFM_REQUIRE(coop, "sfm_bundle_adjust: the device does not support cooperative launches");
    SFM_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ba_solve_kernel, kBaThreads, 0));
    SFM_REQUIRE(per_sm > 0, "sfm_bundle_adjust: the solve kernel cannot be resident");
    const unsigned solve_grid = (unsigned)(sms * std::min(per_sm, 2));

    const BaInputs in{offsets, obs, track_counts, point_status, obs_inlier, X, xy, cams, registered, fixed, max_tracks, max_obs, n_images, S, xy_stride};
    SFM_CUDA_CHECK(cudaMemsetAsync(w.st, 0, sizeof(BaState), st));
    SFM_CUDA_CHECK(cudaMemsetAsync(w.img_used, 0, sizeof(int) * n_images, st));
    const unsigned gt = ba_grid(max_tracks, sms);
    ba_mark_kernel<<<gt, kBaThreads, 0, st>>>(in, w);
    SFM_CUDA_CHECK(cudaGetLastError());
    ba_setup_kernel<<<1, kBaOne, 0, st>>>(in, w);
    SFM_CUDA_CHECK(cudaGetLastError());
    ba_lists_kernel<<<n_images, kBaThreads, 0, st>>>(in, w);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch(3);
    BaInputs in_arg = in;
    BaWork w_arg = w;
    void* solve_args[] = {&in_arg, &w_arg};
    const double ftol = params->function_tolerance, ptol = params->parameter_tolerance;
    for (int it = 0; it < params->max_iters; ++it) {
        ba_point_kernel<<<gt, kBaThreads, 0, st>>>(in, w);
        SFM_CUDA_CHECK(cudaGetLastError());
        ba_camera_kernel<<<n_images, kBaThreads, 0, st>>>(in, w);
        SFM_CUDA_CHECK(cudaGetLastError());
        SFM_CUDA_CHECK(cudaLaunchCooperativeKernel((const void*)ba_solve_kernel, dim3(solve_grid), dim3(kBaThreads), solve_args, 0, st));
        ba_update_kernel<<<gt, kBaThreads, 0, st>>>(in, w);
        SFM_CUDA_CHECK(cudaGetLastError());
        ba_decide_kernel<<<1, kBaOne, 0, st>>>(params->max_iters, ftol, ptol, w);
        SFM_CUDA_CHECK(cudaGetLastError());
        count_launch(5);
    }
    const long long out_work = std::max({12ll * n_images, 3ll * max_tracks, (long long)max_obs});
    ba_output_kernel<<<ba_grid(out_work, sms), kBaThreads, 0, st>>>(in, w, out_pose, out_X, out_obs_error, out_summary);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return SFM_OK;
}
