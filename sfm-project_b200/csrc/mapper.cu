// mapper.cu -- the two device steps of incremental reconstruction that sit between the others.  Compile with -fmad=false.
//
// include/sfm_b200.h, "incremental reconstruction", states the contract.  Three kernels:
//   next_score_kernel    one CTA per image: the image's visible points (features whose track has a point, sfm_pnp_gather's
//                        predicate) set bits of a visibility pyramid in shared memory (atomicOr, so the bits do not depend on
//                        the order); the score sums d^2 * (occupied cells) per level, in int64
//   next_select_kernel   one CTA: every candidate's rank under (score desc, visible desc, image asc) by comparing it with
//                        every other candidate; the first max_select ranks are written and their trials incremented
//   filter_kernel        one warp per track, grid-stride as triangulation: the observations that stay inliers (registered
//                        image, obs_error <= max_error), then a search over their pairs for a triangulation angle of at least
//                        min_angle that stops once any lane has found one (the result is a yes / no, so the scan order does
//                        not matter); statuses 3 and 2 as triangulation writes them
// Integer arithmetic apart from the cell index and the angle, both in fp64 with IEEE basic operations: bit-identical to
// oracle/mapper_oracle.py.
#include <algorithm>

#include "ransac_common.cuh"

namespace sfm {

constexpr int kNextThreads = 256;
constexpr int kMaxLevels = 8;
constexpr int kMaxMapperImages = 1024;  // bundle adjustment's cap
constexpr int kFilterWarps = 4;

// 32-bit words of level l of the pyramid: a d x d grid, d = 2^(l+1), each level starting on a word
static __host__ __device__ constexpr int level_words(int l) { return (4 << (2 * l)) < 32 ? 1 : (4 << (2 * l)) / 32; }
static __host__ __device__ constexpr int pyramid_words(int levels) { return levels == 0 ? 0 : pyramid_words(levels - 1) + level_words(levels - 1); }

__global__ void __launch_bounds__(kNextThreads) next_score_kernel(int S, const int32_t* __restrict__ track_of,
                                                                  const int64_t* __restrict__ track_counts, long long max_tracks,
                                                                  const uint8_t* __restrict__ point_status, const float* __restrict__ xy,
                                                                  int xy_stride, const int32_t* __restrict__ image_size, int levels,
                                                                  int32_t* __restrict__ out_visible, int64_t* __restrict__ out_score)
{
    __shared__ uint32_t bits[pyramid_words(kMaxLevels)];
    __shared__ long long part[kNextThreads / 32];
    __shared__ int vis[kNextThreads / 32];
    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int n_words = 0;
    for (int l = 0; l < levels; ++l) n_words += level_words(l);
    for (int w = tid; w < n_words; w += kNextThreads) bits[w] = 0u;
    __syncthreads();
    const long long n_tracks = min((long long)__ldg(track_counts), max_tracks);
    const double w = (double)__ldg(image_size + 2 * img), h = (double)__ldg(image_size + 2 * img + 1);
    int visible = 0;
    for (int f = tid; f < S; f += kNextThreads) {
        const int k = __ldg(track_of + (long long)img * S + f);
        if (!(k >= 0 && k < n_tracks && __ldg(point_status + k) == 0)) continue;
        ++visible;
        const float2 p = __ldg(reinterpret_cast<const float2*>(xy) + (long long)img * xy_stride + f);
        int off = 0;
        for (int l = 0; l < levels; ++l) {
            const int d = 2 << l;
            double cx = floor((double)p.x * (double)d / w), cy = floor((double)p.y * (double)d / h);
            cx = cx > 0.0 ? (cx < (double)(d - 1) ? cx : (double)(d - 1)) : 0.0;        // NaN -> 0
            cy = cy > 0.0 ? (cy < (double)(d - 1) ? cy : (double)(d - 1)) : 0.0;
            const int cell = (int)cy * d + (int)cx;
            atomicOr(&bits[off + (cell >> 5)], 1u << (cell & 31));
            off += level_words(l);
        }
    }
    __syncthreads();
    long long s = 0;
    int off = 0;
    for (int l = 0; l < levels; ++l) {
        const long long d2 = 4ll << (2 * l);
        for (int i = tid; i < level_words(l); i += kNextThreads) s += d2 * __popc(bits[off + i]);
        off += level_words(l);
    }
    for (int o = 16; o >= 1; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        visible += __shfl_xor_sync(0xffffffffu, visible, o);
    }
    if (lane == 0) { part[warp] = s; vis[warp] = visible; }
    __syncthreads();
    if (tid == 0) {
        long long ts = 0;
        int tv = 0;
        for (int i = 0; i < kNextThreads / 32; ++i) { ts += part[i]; tv += vis[i]; }
        out_visible[img] = tv;
        out_score[img] = ts;
    }
}

__global__ void __launch_bounds__(kMaxMapperImages) next_select_kernel(int n_images, const int32_t* __restrict__ visible,
                                                                       const int64_t* __restrict__ score, const uint8_t* __restrict__ registered,
                                                                       int32_t* __restrict__ trials, sfm_next_images_params prm,
                                                                       int32_t* __restrict__ out_images, int32_t* __restrict__ out_n_selected)
{
    __shared__ long long sc[kMaxMapperImages];
    __shared__ int vi[kMaxMapperImages];
    __shared__ int cand[kMaxMapperImages];
    const int i = threadIdx.x;
    bool c = false;
    if (i < n_images) {
        sc[i] = score[i];
        vi[i] = visible[i];
        c = registered[i] == 0 && trials[i] < prm.max_trials && vi[i] >= prm.min_visible;
        cand[i] = c;
    }
    const int n_cand = __syncthreads_count(c);
    const int n_sel = min(n_cand, prm.max_select);
    if (c) {
        const long long s = sc[i];
        const int v = vi[i];
        int rank = 0;
        for (int j = 0; j < n_images; ++j)
            rank += cand[j] && (sc[j] > s || (sc[j] == s && (vi[j] > v || (vi[j] == v && j < i))));
        if (rank < n_sel) {
            out_images[rank] = i;
            trials[i] += 1;
        }
    }
    for (int r = n_sel + i; r < prm.max_select; r += blockDim.x) out_images[r] = -1;
    if (i == 0) *out_n_selected = n_sel;
}

__global__ void __launch_bounds__(32 * kFilterWarps) filter_kernel(
    int n_images, const int64_t* __restrict__ offsets, const int32_t* __restrict__ obs, const int64_t* __restrict__ track_counts,
    long long max_tracks, const double* __restrict__ cams, const uint8_t* __restrict__ registered, const float* __restrict__ obs_error,
    double max_error, double cos_min, int min_inliers, double* __restrict__ X, int32_t* __restrict__ n_inliers, uint8_t* __restrict__ status,
    uint8_t* obs_inlier, unsigned long long* __restrict__ out_counts)
{
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long n_tracks = min((long long)__ldg(track_counts), max_tracks);
    unsigned long long tally[5] = {0, 0, 0, 0, 0};
    const long long n_warps = (long long)gridDim.x * kFilterWarps;
    for (long long k = (long long)blockIdx.x * kFilterWarps + wib; k < n_tracks; k += n_warps) {
        int st = status[k];
        if (st != 0) {
            if (lane == 0)
#pragma unroll
                for (int s = 0; s < 5; ++s) tally[s] += st == s;
            continue;
        }
        const long long o0 = __ldg(offsets + k);
        const int L = (int)(__ldg(offsets + k + 1) - o0);
        // ---- the observations that stay inliers, written at once (read back by the pair search below)
        int n = 0;
        for (int i = lane; i < L; i += 32) {
            const int img = __ldg(obs + 2 * (o0 + i));
            bool inl = obs_inlier[o0 + i] != 0 && img >= 0 && img < n_images && __ldg(registered + img) != 0;
            inl = inl && (double)obs_error[o0 + i] <= max_error;
            obs_inlier[o0 + i] = inl;
            n += inl;
        }
        for (int o = 16; o >= 1; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
        __syncwarp();                       // every lane's flags are visible to the whole warp
        const double Xk[3] = {X[3 * k], X[3 * k + 1], X[3 * k + 2]};
        if (n < min_inliers) {
            st = 3;
        } else {
            // ---- any pair (a, b), a < b, of inliers whose rays meet at X at min_angle or more; lane owns a = lane + 32 r
            bool found = false;
            for (int a0 = 0; a0 < L && !found; a0 += 32) {
                const int a = a0 + lane;
                bool mine = false;
                if (a < L && obs_inlier[o0 + a]) {
                    Camera A;
                    load_camera(cams + 16ll * __ldg(obs + 2 * (o0 + a)), A);
                    double Ca[3];
                    camera_center(A, Ca);
                    for (int b = a + 1; b < L && !mine; ++b) {
                        if (!obs_inlier[o0 + b]) continue;
                        Camera B;
                        load_camera(cams + 16ll * __ldg(obs + 2 * (o0 + b)), B);
                        double Cb[3];
                        camera_center(B, Cb);
                        mine = ray_cos(Xk, Ca, Cb) <= cos_min;
                    }
                }
                found = __any_sync(0xffffffffu, mine);
            }
            if (!found) st = 2;
        }
        if (st != 0) {
            for (int i = lane; i < L; i += 32) obs_inlier[o0 + i] = 0;
            if (lane < 3) X[3 * k + lane] = 0.0;
        }
        if (lane == 0) {
            n_inliers[k] = st == 2 ? 0 : n;
            status[k] = (uint8_t)st;
#pragma unroll
            for (int s = 0; s < 5; ++s) tally[s] += st == s;
        }
        __syncwarp();
    }
    if (lane == 0)
#pragma unroll
        for (int s = 0; s < 5; ++s)
            if (tally[s]) atomicAdd(&out_counts[s], tally[s]);
}

}  // namespace sfm

using namespace sfm;

extern "C" int sfm_next_images(int n_images, int S, const int32_t* track_of, const int64_t* track_counts, int64_t max_tracks,
                               const uint8_t* point_status, const float* xy, int xy_stride, const int32_t* image_size,
                               const uint8_t* registered, int32_t* trials, const sfm_next_images_params* params, int32_t* out_images,
                               int32_t* out_n_selected, int32_t* out_visible, int64_t* out_score, void* stream)
{
    SFM_REQUIRE(params, "sfm_next_images: NULL params");
    SFM_REQUIRE(track_of && track_counts && point_status && xy && image_size && registered && trials && out_images && out_n_selected &&
                    out_visible && out_score,
                "sfm_next_images: NULL argument");
    SFM_REQUIRE(n_images > 0 && n_images <= kMaxMapperImages, "sfm_next_images: n_images must lie in [1, %d], got %d", kMaxMapperImages,
                n_images);
    SFM_REQUIRE(S > 0 && xy_stride >= S, "sfm_next_images: S = %d must be positive and at most xy_stride = %d", S, xy_stride);
    SFM_REQUIRE(max_tracks >= 0, "sfm_next_images: negative track capacity");
    SFM_REQUIRE(params->levels >= 1 && params->levels <= kMaxLevels, "sfm_next_images: levels must lie in [1, %d], got %d", kMaxLevels,
                params->levels);
    SFM_REQUIRE(params->max_select >= 1, "sfm_next_images: max_select must be positive, got %d", params->max_select);
    SFM_REQUIRE(params->max_trials >= 1, "sfm_next_images: max_trials must be positive, got %d", params->max_trials);
    SFM_REQUIRE(params->min_visible >= 0, "sfm_next_images: min_visible must be non-negative, got %d", params->min_visible);
    cudaStream_t st = (cudaStream_t)stream;
    next_score_kernel<<<n_images, kNextThreads, 0, st>>>(S, track_of, track_counts, max_tracks, point_status, xy, xy_stride, image_size,
                                                         params->levels, out_visible, out_score);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    next_select_kernel<<<1, kMaxMapperImages, 0, st>>>(n_images, out_visible, out_score, registered, trials, *params, out_images,
                                                       out_n_selected);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return SFM_OK;
}

extern "C" int sfm_filter_points(int n_images, const int64_t* offsets, const int32_t* obs, const int64_t* track_counts, int64_t max_tracks,
                                 const double* cams, const uint8_t* registered, const float* obs_error, const sfm_filter_points_params* params,
                                 double* X, int32_t* n_inliers, uint8_t* point_status, uint8_t* obs_inlier, int64_t* out_counts, void* stream)
{
    SFM_REQUIRE(params, "sfm_filter_points: NULL params");
    SFM_REQUIRE(offsets && obs && track_counts && cams && registered && obs_error && X && n_inliers && point_status && obs_inlier && out_counts,
                "sfm_filter_points: NULL argument");
    SFM_REQUIRE(n_images > 0, "sfm_filter_points: n_images must be positive, got %d", n_images);
    SFM_REQUIRE(max_tracks >= 0, "sfm_filter_points: negative track capacity");
    SFM_REQUIRE(params->min_inliers >= 2, "sfm_filter_points: min_inliers must be at least 2, got %d", params->min_inliers);
    SFM_REQUIRE(params->min_angle >= 0.0 && params->min_angle < 90.0, "sfm_filter_points: min_angle must lie in [0, 90) degrees, got %g",
                params->min_angle);
    SFM_REQUIRE(params->max_error >= 0.0 && params->max_error < 1e150, "sfm_filter_points: max_error must be non-negative and finite, got %g",
                params->max_error);
    const double cos_min = cos(params->min_angle * 0.017453292519943295);     // as sfm_triangulate_tracks computes it
    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0, sms = 0;
    SFM_CUDA_CHECK(cudaGetDevice(&dev));
    SFM_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    SFM_CUDA_CHECK(cudaMemsetAsync(out_counts, 0, 5 * sizeof(int64_t), st));
    const long long want = (max_tracks + kFilterWarps - 1) / kFilterWarps;
    const unsigned grid = (unsigned)std::max(1ll, std::min(want, 16ll * sms));
    filter_kernel<<<grid, 32 * kFilterWarps, 0, st>>>(n_images, offsets, obs, track_counts, max_tracks, cams, registered, obs_error,
                                                      params->max_error, cos_min, params->min_inliers, X, n_inliers, point_status,
                                                      obs_inlier, (unsigned long long*)out_counts);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return SFM_OK;
}
