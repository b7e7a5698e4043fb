// triangulate.cu -- robust multi-view triangulation of feature tracks from known cameras.  Compile with -fmad=false.
//
// Every track (tracks.cu) becomes one 3-D point: two-view DLT hypotheses drawn as RANSAC samples, scored by pixel
// reprojection error in every usable view, the best refit by an N-view DLT over its inliers (include/sfm_b200.h,
// "track triangulation", states the contract).  Cameras are x ~ K (R X + t), X in world coordinates.
//
// One warp per track, grid-stride over the worst-case track capacity (the track count is read on the device):
//   stage    the first kTriStage usable observations (registered image, valid index) as (x^, y^, camera) in shared memory;
//            the obs index of every later one goes to the track's slice of obs_error, which is written last
//   sample   lanes own hypotheses: a batch of 32 / 32 / 64 / 128 is 1 / 1 / 2 / 4 per lane (ransac_batch), each scored
//            over every usable view in one pass; argmax by shuffles in hypothesis order, then the adaptive stop rule
//   refit    lane 0 sums the normal matrix over the inliers serially in observation order; the warp recounts
//   emit     per observation inlier flag and reprojection error; per track point, inlier count and status
// fp64 throughout, IEEE basic operations in a fixed order: bit-identical to oracle/triangulate.c.
#include <algorithm>

#include "ransac_common.cuh"

namespace sfm {

constexpr int kTriWarps = 4;           // tracks in flight per CTA
constexpr int kTriStage = 256;         // usable observations per track staged in shared memory
constexpr int kTriPerLane = kBatch / 32;

enum TriStatus { kTriOk = 0, kTriFewViews = 1, kTriNoModel = 2, kTriFewInliers = 3, kTriInvalid = 4, kTriStatuses = 5 };

struct TriStage {
    double2 nxy[kTriStage];
    int cam[kTriStage];
};

struct TriInputs {
    const int32_t* obs;
    const float* xy;
    const double* cams;                 // [n_images, 16] = fx fy cx cy R(9, row-major) t(3)
    const uint8_t* registered;
    int n_images, S, xy_stride;
};

// Normalised coordinates of observation (img, f): x^ = ((double)x - cx) / fx, as pose.cu
static __device__ __forceinline__ void normalised(const TriInputs& in, int img, int f, double& x, double& y)
{
    const float* p = in.xy + 2 * ((long long)img * in.xy_stride + f);
    const double* c = in.cams + 16ll * img;
    x = ((double)__ldg(p) - __ldg(c + 2)) / __ldg(c + 0);
    y = ((double)__ldg(p + 1) - __ldg(c + 3)) / __ldg(c + 1);
}

// The usable observations of one track: u < kTriStage from shared memory, later ones through the obs index map.
struct TriTrack {
    const TriStage* st;
    const int* map;                     // the track's slice of obs_error, as int32 obs indices (u >= kTriStage only)
    long long o0;
    __device__ __forceinline__ void get(const TriInputs& in, int u, int& cam, double& x, double& y) const
    {
        if (u < kTriStage) {
            const double2 v = st->nxy[u];
            x = v.x; y = v.y; cam = st->cam[u];
        } else {
            const long long i = o0 + __ldcg(map + u);
            cam = __ldg(in.obs + 2 * i);
            normalised(in, cam, __ldg(in.obs + 2 * i + 1), x, y);
        }
    }
};

struct Normal {
    double g[10];                       // upper triangle of the 4 x 4 normal matrix, row by row
};

struct Point {
    double x[3];
    int ok;
};

// Adds the two DLT rows of one observation, fx (x^ r3 - r1) and fy (y^ r3 - r2) of [R|t], to the 10 upper-triangle entries
// of the 4 x 4 normal matrix (row x^ first, then row y^).  The focal lengths make each row's residual about a pixel
// residual times the depth, so views of different cameras weigh alike; unscaled rows would weigh a view by about 1/f.
static __device__ __forceinline__ void add_rows(Normal& N, const Camera& K, double x, double y)
{
    double a[4], b[4];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        a[c] = (x * K.r[6 + c] - K.r[0 + c]) * K.fx;
        b[c] = (y * K.r[6 + c] - K.r[3 + c]) * K.fy;
    }
    a[3] = (x * K.t[2] - K.t[0]) * K.fx;
    b[3] = (y * K.t[2] - K.t[1]) * K.fy;
    int e = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) {
            N.g[e] = N.g[e] + a[i] * a[j];
            N.g[e] = N.g[e] + b[i] * b[j];
            ++e;
        }
}

// Eigenvector of the smallest eigenvalue (6 Jacobi sweeps, as pose.cu), de-homogenised; ok = 0 when |w| <= 1e-300.
static __device__ __noinline__ Point solve_point(Normal N)
{
    double G[16], V[16];
    int e = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) {
            G[i * 4 + j] = N.g[e];
            G[j * 4 + i] = N.g[e];
            ++e;
        }
    jacobi_eig_n<4>(G, V, 6);
    int k = 0;
    double gk = G[0];
    if (G[5] < gk) { k = 1; gk = G[5]; }
    if (G[10] < gk) { k = 2; gk = G[10]; }
    if (G[15] < gk) { k = 3; gk = G[15]; }
    const double e0 = k == 0 ? V[0] : k == 1 ? V[1] : k == 2 ? V[2] : V[3];
    const double e1 = k == 0 ? V[4] : k == 1 ? V[5] : k == 2 ? V[6] : V[7];
    const double e2 = k == 0 ? V[8] : k == 1 ? V[9] : k == 2 ? V[10] : V[11];
    const double w = k == 0 ? V[12] : k == 1 ? V[13] : k == 2 ? V[14] : V[15];
    Point P{{0.0, 0.0, 0.0}, 0};
    if (!(fabs(w) > 1e-300)) return P;
    P.x[0] = e0 / w;
    P.x[1] = e1 / w;
    P.x[2] = e2 / w;
    P.ok = 1;
    return P;
}

static __device__ __forceinline__ double depth(const Camera& K, const double* X)
{
    return K.r[6] * X[0] + K.r[7] * X[1] + K.r[8] * X[2] + K.t[2];
}

// Hypothesis `hyp` of track `k`: the DLT point of two usable observations (the earlier one's rows first), kept (ok = 1) iff
// both depths are positive and the ray angle at the point is at least min_angle (cos <= cos_min).
static __device__ __forceinline__ Point hypothesis(const TriInputs& in, const TriTrack& tk, uint64_t seed, uint32_t k, int hyp, int M,
                                                   double cos_min)
{
    int idx[2];
    draw_sample(seed, k, (uint32_t)hyp, 2, M, idx);
    const int ua = min(idx[0], idx[1]), ub = max(idx[0], idx[1]);
    int ca, cb;
    double xa, ya, xb, yb;
    tk.get(in, ua, ca, xa, ya);
    tk.get(in, ub, cb, xb, yb);
    Camera A, B;
    load_camera(in.cams + 16ll * ca, A);
    load_camera(in.cams + 16ll * cb, B);
    Normal N;
#pragma unroll
    for (int e = 0; e < 10; ++e) N.g[e] = 0.0;
    add_rows(N, A, xa, ya);
    add_rows(N, B, xb, yb);
    Point P = solve_point(N);
    if (!P.ok) return P;
    const double* X = P.x;
    double Ca[3], Cb[3];
    camera_center(A, Ca);
    camera_center(B, Cb);
    const double cosang = ray_cos(X, Ca, Cb);
    P.ok = depth(A, X) > 0.0 && depth(B, X) > 0.0 && cosang <= cos_min;
    return P;
}

// Inliers of X over the usable observations, counted by the whole warp (every lane returns the total).
static __device__ int warp_count(const TriInputs& in, const TriTrack& tk, int M, const double* X, double thr2)
{
    int n = 0;
    for (int u = threadIdx.x & 31; u < M; u += 32) {
        int c;
        double x, y, e2;
        tk.get(in, u, c, x, y);
        Camera K;
        load_camera(in.cams + 16ll * c, K);
        n += reproject(K, X, x, y, thr2, e2);
    }
    for (int off = 16; off >= 1; off >>= 1) n += __shfl_xor_sync(0xffffffffu, n, off);
    return n;
}

__global__ void __launch_bounds__(32 * kTriWarps) triangulate_kernel(
    TriInputs in, const int64_t* __restrict__ offsets, const int64_t* __restrict__ track_counts, long long max_tracks,
    sfm_triangulate_params prm, double cos_min, double* __restrict__ out_X, int32_t* __restrict__ out_ninl,
    uint8_t* __restrict__ out_status, uint8_t* __restrict__ out_obs_inlier, float* out_obs_error, unsigned long long* out_counts)
{
    __shared__ TriStage stage[kTriWarps];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    TriStage& S = stage[wib];
    const long long n_tracks = min((long long)__ldg(track_counts), max_tracks);
    const double thr2 = prm.max_error * prm.max_error;
    unsigned long long tally[kTriStatuses] = {0, 0, 0, 0, 0};
    const long long n_warps = (long long)gridDim.x * kTriWarps;
    for (long long k = (long long)blockIdx.x * kTriWarps + wib; k < n_tracks; k += n_warps) {
        const long long o0 = __ldg(offsets + k);
        const int L = (int)(__ldg(offsets + k + 1) - o0);
        int* map = reinterpret_cast<int*>(out_obs_error + o0);
        // ---- stage: validity, the usable observations in obs order
        int M = 0;
        bool bad = false;
        for (int base = 0; base < L; base += 32) {
            const int i = base + lane;
            bool use = false;
            int img = 0, f = 0;
            if (i < L) {
                img = __ldg(in.obs + 2 * (o0 + i));
                f = __ldg(in.obs + 2 * (o0 + i) + 1);
                const bool ok = img >= 0 && img < in.n_images && f >= 0 && f < in.S;
                bad |= !ok;
                use = ok && (!in.registered || __ldg(in.registered + img));
            }
            const unsigned bal = __ballot_sync(0xffffffffu, use);
            const int u = M + __popc(bal & ((1u << lane) - 1u));
            if (use) {
                if (u < kTriStage) {
                    double x, y;
                    normalised(in, img, f, x, y);
                    S.nxy[u] = make_double2(x, y);
                    S.cam[u] = img;
                } else {
                    map[u] = i;
                }
            }
            M += __popc(bal);
        }
        bad = __any_sync(0xffffffffu, bad);
        __syncwarp();
        const TriTrack tk{&S, map, o0};

        int status = kTriOk, cur = 0;
        double X[3] = {0.0, 0.0, 0.0};
        if (bad) {
            status = kTriInvalid;
        } else if (M < 2) {
            status = kTriFewViews;
        } else {
            // ---- sample: hypothesis done + lane + 32 r is lane's r-th of the batch
            int best = -1, done = 0;
            while (done < prm.max_iters) {
                const int nb = min(ransac_batch(done), prm.max_iters - done);
                double hx[kTriPerLane][3];
                int cnt[kTriPerLane];
#pragma unroll
                for (int r = 0; r < kTriPerLane; ++r) {
                    const int h = lane + 32 * r;
                    cnt[r] = -1;
                    hx[r][0] = hx[r][1] = hx[r][2] = 0.0;
                    if (h < nb) {
                        const Point P = hypothesis(in, tk, prm.seed, (uint32_t)k, done + h, M, cos_min);
                        hx[r][0] = P.x[0]; hx[r][1] = P.x[1]; hx[r][2] = P.x[2];
                        cnt[r] = P.ok ? 0 : -1;
                    }
                }
                const int nr = (nb + 31) >> 5;
                for (int u = 0; u < M; ++u) {
                    int c;
                    double x, y, e2;
                    tk.get(in, u, c, x, y);
                    Camera K;
                    load_camera(in.cams + 16ll * c, K);
#pragma unroll
                    for (int r = 0; r < kTriPerLane; ++r)
                        if (r < nr && cnt[r] >= 0) cnt[r] += reproject(K, hx[r], x, y, thr2, e2);
                }
                // strict-greater argmax in hypothesis order: within the lane r ascends, across lanes the smaller index wins ties
                int bc = -1, bh = 0;
#pragma unroll
                for (int r = 0; r < kTriPerLane; ++r)
                    if (cnt[r] > bc) { bc = cnt[r]; bh = lane + 32 * r; }
                for (int off = 16; off >= 1; off >>= 1) {
                    const int oc = __shfl_xor_sync(0xffffffffu, bc, off), oh = __shfl_xor_sync(0xffffffffu, bh, off);
                    if (oc > bc || (oc == bc && oh < bh)) { bc = oc; bh = oh; }
                }
                if (bc > best) {
                    best = bc;
                    const int rr = bh >> 5;
                    double v[3];
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        v[c] = hx[0][c];
#pragma unroll
                        for (int r = 1; r < kTriPerLane; ++r) v[c] = rr == r ? hx[r][c] : v[c];
                        X[c] = __shfl_sync(0xffffffffu, v[c], bh & 31);
                    }
                }
                done += nb;
                if (should_stop(best, M, 2, done, prm.confidence)) break;
            }
            if (best < 0) {
                status = kTriNoModel;
                X[0] = X[1] = X[2] = 0.0;
            } else {
                // ---- refit: N-view DLT over the inliers, kept iff it has at least as many
                cur = best;
                for (int round = 0; round < kLoRounds && cur >= 2; ++round) {
                    Point R{{0.0, 0.0, 0.0}, 0};
                    if (lane == 0) {
                        Normal N;
#pragma unroll
                        for (int e = 0; e < 10; ++e) N.g[e] = 0.0;
                        for (int u = 0; u < M; ++u) {
                            int c;
                            double x, y, e2;
                            tk.get(in, u, c, x, y);
                            Camera K;
                            load_camera(in.cams + 16ll * c, K);
                            if (reproject(K, X, x, y, thr2, e2)) add_rows(N, K, x, y);
                        }
                        R = solve_point(N);
                    }
                    if (!__shfl_sync(0xffffffffu, R.ok, 0)) break;
                    double Xr[3];
#pragma unroll
                    for (int c = 0; c < 3; ++c) Xr[c] = __shfl_sync(0xffffffffu, R.x[c], 0);
                    const int n = warp_count(in, tk, M, Xr, thr2);
                    if (n < cur) break;
                    cur = n;
                    X[0] = Xr[0]; X[1] = Xr[1]; X[2] = Xr[2];
                }
                if (cur < prm.min_inliers) {
                    status = kTriFewInliers;
                    X[0] = X[1] = X[2] = 0.0;
                }
            }
        }
        __syncwarp();                       // every map read is done: obs_error may be written
        // ---- emit
        for (int i = lane; i < L; i += 32) {
            float err = __int_as_float(0x7fc00000);
            uint8_t inl = 0;
            if (status == kTriOk) {
                const int img = __ldg(in.obs + 2 * (o0 + i));
                if (!in.registered || __ldg(in.registered + img)) {
                    double x, y, e2;
                    normalised(in, img, __ldg(in.obs + 2 * (o0 + i) + 1), x, y);
                    Camera K;
                    load_camera(in.cams + 16ll * img, K);
                    inl = reproject(K, X, x, y, thr2, e2);
                    err = (float)sqrt(e2);
                }
            }
            out_obs_inlier[o0 + i] = inl;
            out_obs_error[o0 + i] = err;
        }
        if (lane < 3) out_X[3 * k + lane] = lane == 0 ? X[0] : lane == 1 ? X[1] : X[2];
        if (lane == 0) {
            out_ninl[k] = (status == kTriOk || status == kTriFewInliers) ? cur : 0;
            out_status[k] = (uint8_t)status;
            tally[status] += 1;
        }
        __syncwarp();                       // the stage is rewritten by the warp's next track
    }
    if (lane == 0)
        for (int s = 0; s < kTriStatuses; ++s)
            if (tally[s]) atomicAdd(&out_counts[s], tally[s]);
}

}  // namespace sfm

using namespace sfm;

extern "C" int sfm_triangulate_tracks(int n_images, int S, const int64_t* offsets, const int32_t* obs, const int64_t* track_counts,
                                      int64_t max_tracks, const float* xy, int xy_stride, const double* cams, const uint8_t* registered,
                                      const sfm_triangulate_params* params, double* out_X, int32_t* out_n_inliers, uint8_t* out_status,
                                      uint8_t* out_obs_inlier, float* out_obs_error, int64_t* out_counts, void* stream)
{
    SFM_REQUIRE(params, "sfm_triangulate_tracks: NULL params");
    SFM_REQUIRE(offsets && obs && track_counts && xy && cams && out_X && out_n_inliers && out_status && out_obs_inlier && out_obs_error &&
                    out_counts,
                "sfm_triangulate_tracks: NULL argument");
    SFM_REQUIRE(n_images > 0 && S > 0, "sfm_triangulate_tracks: n_images and S must be positive");
    SFM_REQUIRE((long long)n_images * S < (1ll << 31), "sfm_triangulate_tracks: n_images * S = %lld must stay below 2^31",
                (long long)n_images * S);
    SFM_REQUIRE(xy_stride >= S, "sfm_triangulate_tracks: xy_stride %d is below S = %d", xy_stride, S);
    SFM_REQUIRE(max_tracks >= 0, "sfm_triangulate_tracks: negative track capacity");
    SFM_REQUIRE(params->max_iters > 0, "sfm_triangulate_tracks: max_iters must be positive, got %d", params->max_iters);
    SFM_REQUIRE(params->min_inliers >= 2, "sfm_triangulate_tracks: min_inliers must be at least 2, got %d", params->min_inliers);
    SFM_REQUIRE(params->min_angle >= 0.0 && params->min_angle < 90.0, "sfm_triangulate_tracks: min_angle must lie in [0, 90) degrees, got %g",
                params->min_angle);
    SFM_REQUIRE(params->max_error > 0.0 && params->max_error < 1e150, "sfm_triangulate_tracks: max_error must be positive and finite, got %g",
                params->max_error);
    const double cos_min = cos(params->min_angle * 0.017453292519943295);     // computed once, as oracle/triangulate.c does
    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0, sms = 0;
    SFM_CUDA_CHECK(cudaGetDevice(&dev));
    SFM_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    SFM_CUDA_CHECK(cudaMemsetAsync(out_counts, 0, kTriStatuses * sizeof(int64_t), st));
    const TriInputs in{obs, xy, cams, registered, n_images, S, xy_stride};
    const long long want = (max_tracks + kTriWarps - 1) / kTriWarps;
    const unsigned grid = (unsigned)std::max(1ll, std::min(want, 16ll * sms));
    triangulate_kernel<<<grid, 32 * kTriWarps, 0, st>>>(in, offsets, track_counts, max_tracks, *params, cos_min, out_X, out_n_inliers,
                                                         out_status, out_obs_inlier, out_obs_error, (unsigned long long*)out_counts);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return SFM_OK;
}
