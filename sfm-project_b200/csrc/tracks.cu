// tracks.cu -- feature tracks from the verified matches (f5).
//
// A track is the set of (image, feature) observations of one scene point, joined through the verified matches: the
// output of correspondence search that registration and multi-view triangulation read (Schoenberger & Frahm 2016, §2.1).
// The reference leaves it to the empty code/3d_reconstruction.py (imported at code/pipeline.py:4); the match rows it
// would read are the `pair_matches` of code/pipeline.py:43-47.
//
// Node n = image * S + feature.  Every used row (q, t) of pair (i, j) is the edge (i*S + q, j*S + t).  Integer work only:
//   hook      one warp per pair strides over its rows; lock-free union with link-by-index (the larger root is CAS'd to
//             point at the smaller one; find halves the path).  parent[x] <= x holds at every step, so once every edge is
//             in, the only root of a component is its minimum node, whatever the interleaving: labels are deterministic.
//   finalize  compress + size per root -> scan over roots (candidate ids and slice offsets in ascending min-node order) ->
//             atomic placement -> per-slice sort (one warp up to 32 observations; one CTA above: 4096-entry shared-memory
//             tiles, then in-CTA merge passes in global memory) + conflict flag -> scan over kept candidates -> final copy and
//             track_of.
// The workspace is caller-owned; nothing synchronises with the host.
#include <limits.h>

#include <algorithm>

#include "common.cuh"

namespace sfm {

void launch_offsets_scan(const int32_t* cnt, int n, int32_t* offset, cudaStream_t st);

constexpr int kScanBlock = 1024;   // items per block of the two-level scans
constexpr int kTile = 4096;        // shared-memory sort tile of the CTA path
constexpr int kWarpMax = 32;       // longest slice the warp path sorts

enum TrackCounter { kInvalid = 0, kConflicting = 1, kShort = 2, kListLen = 3, kCounters = 4 };

struct TrackWorkspace {
    int32_t *parent, *size, *cid, *cstart, *keep, *tid, *tmp, *tmp2, *list;
    int32_t *blk[4], *off[4];      // per-block sums and their scans: [0, 1] over nodes (roots, observations), [2, 3] over candidates
    unsigned long long* counters;
    uint8_t* used;
    size_t bytes;
};

// Section layout of the workspace for N = n_images * S nodes (all sections 256-byte aligned).
static TrackWorkspace carve(uint8_t* base, long long N)
{
    const long long nb = (N + kScanBlock - 1) / kScanBlock;
    TrackWorkspace w{};
    size_t o = 0;
    auto take = [&](long long bytes) {
        uint8_t* p = base + o;
        o = (size_t)align_up(o + bytes, 256);
        return p;
    };
    w.parent = (int32_t*)take(4 * N);
    w.size = (int32_t*)take(4 * N);
    w.cid = (int32_t*)take(4 * N);
    w.cstart = (int32_t*)take(4 * (N + 1));
    w.keep = (int32_t*)take(4 * N);
    w.tid = (int32_t*)take(4 * N);
    w.tmp = (int32_t*)take(4 * N);
    w.tmp2 = (int32_t*)take(4 * N);
    w.list = (int32_t*)take(4 * N);
    for (int k = 0; k < 4; ++k) {
        w.blk[k] = (int32_t*)take(4 * nb);
        w.off[k] = (int32_t*)take(4 * (nb + 1));
    }
    w.counters = (unsigned long long*)take(8 * kCounters);
    w.used = take(N);
    w.bytes = o;
    return w;
}

// ------------------------------------------------------------------ union-find (parent[x] <= x always)
__device__ __forceinline__ int find_root(volatile int32_t* parent, int x)
{
    int cur = parent[x];
    if (cur != x) {
        int prev = x, next;
        while (cur > (next = parent[cur])) {
            parent[prev] = next;            // path halving: prev skips to an ancestor
            prev = cur;
            cur = next;
        }
    }
    return cur;
}

__device__ __forceinline__ void unite(int32_t* parent, int a, int b)
{
    int ra = find_root(parent, a), rb = find_root(parent, b);
    while (ra != rb) {
        // link by index: the larger root is made to point at the smaller; a failed CAS returns a smaller ancestor to retry from
        if (ra < rb) {
            const int old = atomicCAS(&parent[rb], rb, ra);
            if (old == rb) break;
            rb = old;
        } else {
            const int old = atomicCAS(&parent[ra], ra, rb);
            if (old == ra) break;
            ra = old;
        }
    }
}

__global__ void __launch_bounds__(256) tracks_init_kernel(int32_t* __restrict__ parent, uint8_t* __restrict__ used, int N)
{
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n < N) {
        parent[n] = n;
        used[n] = 0;
    }
}

// One warp per pair.  A row is used when its pair has enough inliers, its flag is set and both feature indices lie in [0, S);
// rows that would be used but point outside [0, S) (or belong to a pair naming an image outside [0, n_images)) are counted.
__global__ void __launch_bounds__(256) tracks_hook_kernel(const int32_t* __restrict__ pairs, int n_pairs,
                                                         const int64_t* __restrict__ row_start, const int32_t* __restrict__ n_rows,
                                                         const int32_t* __restrict__ rows, const uint8_t* __restrict__ flag,
                                                         const int32_t* __restrict__ n_inl, int min_pair_inl, int n_images, int S,
                                                         int32_t* parent, uint8_t* used, unsigned long long* counters)
{
    const int p = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= n_pairs) return;
    if (n_inl && n_inl[p] < min_pair_inl) return;
    const int i = pairs[2 * p], j = pairs[2 * p + 1];
    const bool pair_ok = i >= 0 && i < n_images && j >= 0 && j < n_images;
    const int n = n_rows[p];
    const long long s = row_start[p];
    int bad = 0;
    for (int r = lane; r < n; r += 32) {
        const long long k = s + r;
        if (flag && !flag[k]) continue;
        const int q = rows[3 * k], t = rows[3 * k + 1];
        if (!pair_ok || q < 0 || q >= S || t < 0 || t >= S) {
            ++bad;
            continue;
        }
        const int a = i * S + q, b = j * S + t;
        used[a] = 1;
        used[b] = 1;
        unite(parent, a, b);
    }
    for (int o = 16; o; o >>= 1) bad += __shfl_xor_sync(0xffffffffu, bad, o);
    if (lane == 0 && bad) atomicAdd(&counters[kInvalid], (unsigned long long)bad);
}

// Every node points at its root; every used node adds one to its root's size.  The walk halves the path it takes, with
// atomicMin: a pointer only ever moves to a smaller node, i.e. further up, so a halving step can never undo another thread's
// root pointer.  (A union order that no find walks -- edges (k, k+1) arriving with k descending -- leaves a chain as deep as
// its component; the halving here is what keeps the concurrent walks of such a chain short.)
__global__ void __launch_bounds__(256) tracks_compress_kernel(int32_t* parent, const uint8_t* __restrict__ used,
                                                             int32_t* __restrict__ size, int N)
{
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const volatile int32_t* vp = parent;
    int prev = n, cur = vp[n], next;
    while (cur > (next = vp[cur])) {
        atomicMin(&parent[prev], next);
        prev = cur;
        cur = next;
    }
    atomicMin(&parent[n], cur);
    if (used[n]) atomicAdd(&size[cur], 1);
}

// Exclusive scan of two quantities over a 1024-thread block; returns the totals in *tot_a / *tot_b.
__device__ __forceinline__ void block_scan2(int a, int b, int* ex_a, int* ex_b, int* tot_a, int* tot_b)
{
    __shared__ int wa[32], wb[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int sa = a, sb = b;
    for (int o = 1; o < 32; o <<= 1) {
        const int ua = __shfl_up_sync(0xffffffffu, sa, o), ub = __shfl_up_sync(0xffffffffu, sb, o);
        if (lane >= o) sa += ua, sb += ub;
    }
    if (lane == 31) wa[warp] = sa, wb[warp] = sb;
    __syncthreads();
    if (warp == 0) {
        int xa = wa[lane], xb = wb[lane];
        for (int o = 1; o < 32; o <<= 1) {
            const int ua = __shfl_up_sync(0xffffffffu, xa, o), ub = __shfl_up_sync(0xffffffffu, xb, o);
            if (lane >= o) xa += ua, xb += ub;
        }
        wa[lane] = xa, wb[lane] = xb;
    }
    __syncthreads();
    *ex_a = (warp ? wa[warp - 1] : 0) + sa - a;
    *ex_b = (warp ? wb[warp - 1] : 0) + sb - b;
    *tot_a = wa[31];
    *tot_b = wb[31];
}

// Two-level scans.  kRoots: items are nodes; a = "is the root of a candidate", b = its size.  Otherwise items are candidates
// (ascending min node); a = kept, b = its length when kept.  !kApply: per-block totals.  kApply: the exclusive scans plus the
// scanned block offsets give candidate ids / slice starts (kRoots) or track ids / output offsets.
template <bool kRoots, bool kApply>
__global__ void __launch_bounds__(kScanBlock) tracks_scan_kernel(TrackWorkspace w, int N, int64_t* __restrict__ offsets_out)
{
    const int i = blockIdx.x * kScanBlock + threadIdx.x;
    int a = 0, b = 0;
    if (kRoots) {
        if (i < N && w.parent[i] == i && w.size[i] > 0) a = 1, b = w.size[i];
    } else {
        const int n_cand = w.off[0][gridDim.x];
        if (i < n_cand && w.keep[i]) a = 1, b = w.cstart[i + 1] - w.cstart[i];
    }
    int ea, eb, ta, tb;
    block_scan2(a, b, &ea, &eb, &ta, &tb);
    const int k0 = kRoots ? 0 : 2;
    if (!kApply) {
        if (threadIdx.x == 0) w.blk[k0][blockIdx.x] = ta, w.blk[k0 + 1][blockIdx.x] = tb;
        return;
    }
    const int c = w.off[k0][blockIdx.x] + ea, o = w.off[k0 + 1][blockIdx.x] + eb;
    if (kRoots) {
        if (a) {
            w.cid[i] = c;
            w.cstart[c] = o;
            if (b > kWarpMax) w.list[atomicAdd(&w.counters[kListLen], 1ull)] = c;
        }
        if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) w.cstart[w.off[0][gridDim.x]] = w.off[1][gridDim.x];
    } else {
        const int n_cand = w.off[0][gridDim.x];
        if (i < n_cand) w.tid[i] = a ? c : -1;
        if (a) offsets_out[c] = o;
        if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) offsets_out[w.off[2][gridDim.x]] = w.off[3][gridDim.x];
    }
}

// Atomic placement of every used node into its candidate's slice (the size counts down as the cursor).
__global__ void __launch_bounds__(256) tracks_scatter_kernel(TrackWorkspace w, int N)
{
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N || !w.used[n]) return;
    const int r = w.parent[n];
    const int pos = atomicSub(&w.size[r], 1) - 1;
    w.tmp[w.cstart[w.cid[r]] + pos] = n;
}

__device__ __forceinline__ bool keep_candidate(bool conflict, int len, int min_length, int keep_conflicts, int* n_conf, int* n_short)
{
    if (conflict) {
        ++*n_conf;
        if (!keep_conflicts) return false;
    }
    if (len < min_length) {
        ++*n_short;
        return false;
    }
    return true;
}

// Slices of at most 32 observations: one warp each, rank sort (nodes are distinct) and the same-image test on the way.
__global__ void __launch_bounds__(256) tracks_sort_warp_kernel(TrackWorkspace w, int n_blocks, int S, int min_length, int keep_conflicts)
{
    const int lane = threadIdx.x & 31;
    const int n_cand = w.off[0][n_blocks];
    int n_conf = 0, n_short = 0;
    for (int c = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5); c < n_cand; c += (gridDim.x * blockDim.x) >> 5) {
        const int s = w.cstart[c], len = w.cstart[c + 1] - s;
        if (len > kWarpMax) continue;
        const int v = lane < len ? w.tmp[s + lane] : INT_MAX;
        const int img = lane < len ? v / S : -1 - lane;
        int rank = 0;
        bool dup = false;
        for (int k = 0; k < 32; ++k) {
            const int u = __shfl_sync(0xffffffffu, v, k), ui = __shfl_sync(0xffffffffu, img, k);
            rank += u < v;
            dup |= k != lane && ui == img;
        }
        if (lane < len) w.tmp[s + rank] = v;
        const bool conflict = __any_sync(0xffffffffu, dup);
        if (lane == 0) w.keep[c] = keep_candidate(conflict, len, min_length, keep_conflicts, &n_conf, &n_short);
    }
    if (lane == 0 && n_conf) atomicAdd(&w.counters[kConflicting], (unsigned long long)n_conf);
    if (lane == 0 && n_short) atomicAdd(&w.counters[kShort], (unsigned long long)n_short);
}

// Slices above 32 observations (listed by the root scan): one CTA each.  Bitonic sort of 4096-entry tiles in shared memory,
// then merge passes that double the sorted run length (each element finds its place in the partner run by binary search;
// the nodes are distinct), ping-ponging between tmp and tmp2; then the same-image test on adjacent observations.
__global__ void __launch_bounds__(1024) tracks_sort_cta_kernel(TrackWorkspace w, int S, int min_length, int keep_conflicts)
{
    __shared__ int tile[kTile];
    const int n_list = (int)w.counters[kListLen];
    int n_conf = 0, n_short = 0;
    for (int k = blockIdx.x; k < n_list; k += gridDim.x) {
        const int c = w.list[k];
        const int s = w.cstart[c], len = w.cstart[c + 1] - s;
        for (int t0 = 0; t0 < len; t0 += kTile) {
            const int m = min(kTile, len - t0);
            int m2 = 1;
            while (m2 < m) m2 <<= 1;
            for (int x = threadIdx.x; x < m2; x += blockDim.x) tile[x] = x < m ? w.tmp[s + t0 + x] : INT_MAX;
            __syncthreads();
            for (int kk = 2; kk <= m2; kk <<= 1) {
                for (int jj = kk >> 1; jj > 0; jj >>= 1) {
                    for (int x = threadIdx.x; x < m2; x += blockDim.x) {
                        const int y = x ^ jj;
                        if (y > x) {
                            const int a = tile[x], b = tile[y];
                            if (((x & kk) == 0) == (a > b)) tile[x] = b, tile[y] = a;
                        }
                    }
                    __syncthreads();
                }
            }
            for (int x = threadIdx.x; x < m; x += blockDim.x) w.tmp[s + t0 + x] = tile[x];
            __syncthreads();
        }
        int* src = w.tmp + s;
        int* dst = w.tmp2 + s;
        for (int run = kTile; run < len; run <<= 1) {
            for (int x = threadIdx.x; x < len; x += blockDim.x) {
                const int r = x / run;
                const int pb = min((r ^ 1) * run, len), pe = min(pb + run, len);
                const int v = src[x];
                int lo = pb, hi = pe;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (src[mid] < v) lo = mid + 1;
                    else hi = mid;
                }
                dst[(r & ~1) * run + (x - r * run) + (lo - pb)] = v;
            }
            __syncthreads();
            int* t = src;
            src = dst;
            dst = t;
        }
        bool dup = false;
        for (int x = threadIdx.x; x < len; x += blockDim.x) {
            const int v = src[x];
            if (src != w.tmp + s) w.tmp[s + x] = v;
            dup |= x + 1 < len && v / S == src[x + 1] / S;
        }
        const bool conflict = __syncthreads_or(dup);
        if (threadIdx.x == 0) w.keep[c] = keep_candidate(conflict, len, min_length, keep_conflicts, &n_conf, &n_short);
        __syncthreads();
    }
    if (threadIdx.x == 0 && n_conf) atomicAdd(&w.counters[kConflicting], (unsigned long long)n_conf);
    if (threadIdx.x == 0 && n_short) atomicAdd(&w.counters[kShort], (unsigned long long)n_short);
}

// Final copy: observation i of the sorted candidate slices goes to its track's output slice, and track_of names its track.
__global__ void __launch_bounds__(256) tracks_emit_kernel(TrackWorkspace w, int n_blocks, int S, const int64_t* __restrict__ offsets,
                                                         int32_t* __restrict__ obs, int32_t* __restrict__ track_of)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= w.off[1][n_blocks]) return;
    const int n = w.tmp[i];
    const int c = w.cid[w.parent[n]];
    const int t = w.tid[c];
    if (t < 0) return;
    const long long o = offsets[t] + (i - w.cstart[c]);
    obs[2 * o] = n / S;
    obs[2 * o + 1] = n % S;
    track_of[n] = t;
}

__global__ void tracks_counts_kernel(TrackWorkspace w, int n_blocks, int64_t* __restrict__ counts)
{
    counts[0] = w.off[2][n_blocks];                     // tracks
    counts[1] = w.off[3][n_blocks];                     // observations
    counts[2] = (int64_t)w.counters[kConflicting];
    counts[3] = (int64_t)w.counters[kShort];
    counts[4] = (int64_t)w.counters[kInvalid];
}

static int check_sizes(const char* fn, int n_images, int S, const void* workspace, size_t workspace_bytes, TrackWorkspace* w)
{
    SFM_REQUIRE(n_images > 0 && S > 0, "%s: n_images and S must be positive", fn);
    SFM_REQUIRE((long long)n_images * S < (1ll << 31), "%s: n_images * S = %lld nodes must stay below 2^31", fn, (long long)n_images * S);
    SFM_REQUIRE(workspace, "%s: NULL workspace", fn);
    SFM_REQUIRE(((uintptr_t)workspace & 255) == 0, "%s: workspace must be 256-byte aligned", fn);
    *w = carve((uint8_t*)workspace, (long long)n_images * S);
    SFM_REQUIRE(workspace_bytes >= w->bytes, "%s: workspace of %zu bytes, %zu needed", fn, workspace_bytes, w->bytes);
    return SFM_OK;
}

static int check_params(const char* fn, const sfm_track_params* prm)
{
    SFM_REQUIRE(prm, "%s: NULL params", fn);
    SFM_REQUIRE(prm->min_length >= 2, "%s: min_length must be at least 2, got %d", fn, prm->min_length);
    SFM_REQUIRE(prm->keep_conflicts == 0 || prm->keep_conflicts == 1, "%s: keep_conflicts must be 0 or 1", fn);
    return SFM_OK;
}

static unsigned blocks_for(long long n, int per) { return (unsigned)((n + per - 1) / per); }

}  // namespace sfm

using namespace sfm;

extern "C" int sfm_tracks_workspace_bytes(int n_images, int S, size_t* out_bytes)
{
    SFM_REQUIRE(out_bytes, "sfm_tracks_workspace_bytes: NULL argument");
    SFM_REQUIRE(n_images > 0 && S > 0, "sfm_tracks_workspace_bytes: n_images and S must be positive");
    SFM_REQUIRE((long long)n_images * S < (1ll << 31), "sfm_tracks_workspace_bytes: n_images * S = %lld nodes must stay below 2^31",
                (long long)n_images * S);
    *out_bytes = carve(nullptr, (long long)n_images * S).bytes;
    return SFM_OK;
}

extern "C" int sfm_tracks_init(int n_images, int S, void* workspace, size_t workspace_bytes, void* stream)
{
    TrackWorkspace w;
    int rc = check_sizes("sfm_tracks_init", n_images, S, workspace, workspace_bytes, &w);
    if (rc) return rc;
    const int N = n_images * S;
    cudaStream_t st = (cudaStream_t)stream;
    SFM_CUDA_CHECK(cudaMemsetAsync(&w.counters[kInvalid], 0, sizeof(unsigned long long), st));
    tracks_init_kernel<<<blocks_for(N, 256), 256, 0, st>>>(w.parent, w.used, N);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return SFM_OK;
}

extern "C" int sfm_tracks_hook(int n_images, int S, const int32_t* pairs, int n_pairs, const int64_t* row_start, const int32_t* n_rows,
                               const int32_t* rows, const uint8_t* row_flag, const int32_t* n_inliers, const sfm_track_params* params,
                               void* workspace, size_t workspace_bytes, void* stream)
{
    TrackWorkspace w;
    int rc = check_sizes("sfm_tracks_hook", n_images, S, workspace, workspace_bytes, &w);
    if (rc) return rc;
    rc = check_params("sfm_tracks_hook", params);
    if (rc) return rc;
    SFM_REQUIRE(n_pairs >= 0, "sfm_tracks_hook: negative pair count");
    if (n_pairs == 0) return SFM_OK;
    SFM_REQUIRE(pairs && row_start && n_rows && rows, "sfm_tracks_hook: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    tracks_hook_kernel<<<blocks_for(32ll * n_pairs, 256), 256, 0, st>>>(pairs, n_pairs, row_start, n_rows, rows, row_flag, n_inliers,
                                                                        params->min_pair_inliers, n_images, S, w.parent, w.used,
                                                                        w.counters);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return SFM_OK;
}

extern "C" int sfm_tracks_finalize(int n_images, int S, const sfm_track_params* params, void* workspace, size_t workspace_bytes,
                                   int32_t* track_of, int64_t* offsets, int32_t* obs, int64_t* counts, void* stream)
{
    TrackWorkspace w;
    int rc = check_sizes("sfm_tracks_finalize", n_images, S, workspace, workspace_bytes, &w);
    if (rc) return rc;
    rc = check_params("sfm_tracks_finalize", params);
    if (rc) return rc;
    SFM_REQUIRE(track_of && offsets && obs && counts, "sfm_tracks_finalize: NULL argument");
    const int N = n_images * S;
    const int nb = (int)blocks_for(N, kScanBlock);
    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0, sms = 0;
    SFM_CUDA_CHECK(cudaGetDevice(&dev));
    SFM_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    SFM_CUDA_CHECK(cudaMemsetAsync(w.size, 0, 4ull * N, st));
    SFM_CUDA_CHECK(cudaMemsetAsync(&w.counters[kConflicting], 0, 3 * sizeof(unsigned long long), st));
    SFM_CUDA_CHECK(cudaMemsetAsync(track_of, 0xFF, 4ull * N, st));
    tracks_compress_kernel<<<blocks_for(N, 256), 256, 0, st>>>(w.parent, w.used, w.size, N);
    tracks_scan_kernel<true, false><<<nb, kScanBlock, 0, st>>>(w, N, nullptr);
    launch_offsets_scan(w.blk[0], nb, w.off[0], st);
    launch_offsets_scan(w.blk[1], nb, w.off[1], st);
    tracks_scan_kernel<true, true><<<nb, kScanBlock, 0, st>>>(w, N, nullptr);
    tracks_scatter_kernel<<<blocks_for(N, 256), 256, 0, st>>>(w, N);
    tracks_sort_warp_kernel<<<(unsigned)std::min<long long>(blocks_for(N, 256), 16ll * sms), 256, 0, st>>>(w, nb, S, params->min_length,
                                                                                                           params->keep_conflicts);
    tracks_sort_cta_kernel<<<2 * sms, 1024, 0, st>>>(w, S, params->min_length, params->keep_conflicts);
    tracks_scan_kernel<false, false><<<nb, kScanBlock, 0, st>>>(w, N, nullptr);
    launch_offsets_scan(w.blk[2], nb, w.off[2], st);
    launch_offsets_scan(w.blk[3], nb, w.off[3], st);
    tracks_scan_kernel<false, true><<<nb, kScanBlock, 0, st>>>(w, N, offsets);
    tracks_emit_kernel<<<blocks_for(N, 256), 256, 0, st>>>(w, nb, S, offsets, obs, track_of);
    tracks_counts_kernel<<<1, 1, 0, st>>>(w, nb, counts);
    SFM_CUDA_CHECK(cudaGetLastError());
    count_launch(10);                                   // (the four scans are counted by launch_offsets_scan)
    return SFM_OK;
}
