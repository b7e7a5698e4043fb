/* triangulate.c -- CPU oracle for the robust multi-view triangulation of feature tracks (sfm_triangulate_tracks).
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under sfm-project_b200/ links, imports or executes this file; only tests/ and
 * tools/ may.
 *
 * What it restates: the contract of include/sfm_b200.h, "track triangulation", serially -- one track after another,
 * hypotheses in index order (strict-greater selection, so the earlier of two equal counts wins, as the kernel's
 * in-order argmax does), the normal matrices summed in observation order.  Operation for operation the same as
 * sfm-project_b200/csrc/triangulate.cu; built with -ffp-contract=off so points, counts, flags and errors are compared
 * bit for bit.  Sampling, the stop rule and the Jacobi solver come from ransac_common.h.
 */
#include "ransac_common.h"

typedef struct {
    double fx, fy, r[9], t[3];
} tri_camera;

static void tri_load_camera(const double* c, tri_camera* K)
{
    K->fx = c[0];
    K->fy = c[1];
    for (int i = 0; i < 9; ++i) K->r[i] = c[4 + i];
    for (int i = 0; i < 3; ++i) K->t[i] = c[13 + i];
}

static void tri_add_rows(double G[10], const tri_camera* K, double x, double y)
{
    double a[4], b[4];
    for (int c = 0; c < 3; ++c) {
        a[c] = x * K->r[6 + c] - K->r[0 + c];
        b[c] = y * K->r[6 + c] - K->r[3 + c];
    }
    a[3] = x * K->t[2] - K->t[0];
    b[3] = y * K->t[2] - K->t[1];
    int e = 0;
    for (int i = 0; i < 4; ++i)
        for (int j = i; j < 4; ++j) {
            G[e] = G[e] + a[i] * a[j];
            G[e] = G[e] + b[i] * b[j];
            ++e;
        }
}

static int tri_solve(const double G10[10], double X[3])
{
    double G[16], V[16];
    int e = 0;
    for (int i = 0; i < 4; ++i)
        for (int j = i; j < 4; ++j) {
            G[i * 4 + j] = G10[e];
            G[j * 4 + i] = G10[e];
            ++e;
        }
    jacobi_eig(G, V, 4, 6);
    int k = 0;
    for (int j = 1; j < 4; ++j)
        if (G[j * 5] < G[k * 5]) k = j;
    double w = V[12 + k];
    X[0] = 0.0; X[1] = 0.0; X[2] = 0.0;
    if (!(fabs(w) > 1e-300)) return 0;
    X[0] = V[0 + k] / w;
    X[1] = V[4 + k] / w;
    X[2] = V[8 + k] / w;
    return 1;
}

static double tri_depth(const tri_camera* K, const double* X)
{
    return K->r[6] * X[0] + K->r[7] * X[1] + K->r[8] * X[2] + K->t[2];
}

static int tri_reproject(const tri_camera* K, const double* X, double x, double y, double thr2, double* e2)
{
    double p0 = K->r[0] * X[0] + K->r[1] * X[1] + K->r[2] * X[2] + K->t[0];
    double p1 = K->r[3] * X[0] + K->r[4] * X[1] + K->r[5] * X[2] + K->t[1];
    double p2 = K->r[6] * X[0] + K->r[7] * X[1] + K->r[8] * X[2] + K->t[2];
    if (!(p2 > 0.0)) {
        *e2 = INFINITY;
        return 0;
    }
    double iz = 1.0 / p2;
    double ex = (p0 * iz - x) * K->fx;
    double ey = (p1 * iz - y) * K->fy;
    *e2 = ex * ex + ey * ey;
    return *e2 <= thr2;
}

static void tri_center(const tri_camera* K, double* C)
{
    for (int i = 0; i < 3; ++i) C[i] = -(K->r[i] * K->t[0] + K->r[3 + i] * K->t[1] + K->r[6 + i] * K->t[2]);
}

typedef struct {
    const double* cams;
    const int* cam;          /* [M] camera of each usable observation */
    const double* nx;        /* [M] normalised coordinates            */
    const double* ny;
    int M;
    double thr2;
} tri_track;

static int tri_count(const tri_track* T, const double* X)
{
    int n = 0;
    for (int u = 0; u < T->M; ++u) {
        tri_camera K;
        double e2;
        tri_load_camera(T->cams + 16 * (size_t)T->cam[u], &K);
        n += tri_reproject(&K, X, T->nx[u], T->ny[u], T->thr2, &e2);
    }
    return n;
}

static int tri_hypothesis(const tri_track* T, uint64_t seed, uint32_t k, int hyp, double cos_min, double* X)
{
    int idx[2];
    draw_sample(seed, k, (uint32_t)hyp, 2, T->M, idx);
    int ua = idx[0] < idx[1] ? idx[0] : idx[1];
    int ub = idx[0] < idx[1] ? idx[1] : idx[0];
    tri_camera A, B;
    tri_load_camera(T->cams + 16 * (size_t)T->cam[ua], &A);
    tri_load_camera(T->cams + 16 * (size_t)T->cam[ub], &B);
    double G[10] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    tri_add_rows(G, &A, T->nx[ua], T->ny[ua]);
    tri_add_rows(G, &B, T->nx[ub], T->ny[ub]);
    if (!tri_solve(G, X)) return 0;
    double Ca[3], Cb[3];
    tri_center(&A, Ca);
    tri_center(&B, Cb);
    double da0 = X[0] - Ca[0], da1 = X[1] - Ca[1], da2 = X[2] - Ca[2];
    double db0 = X[0] - Cb[0], db1 = X[1] - Cb[1], db2 = X[2] - Cb[2];
    double dot = da0 * db0 + da1 * db1 + da2 * db2;
    double na = da0 * da0 + da1 * da1 + da2 * da2;
    double nb = db0 * db0 + db1 * db1 + db2 * db2;
    double cosang = dot / sqrt(na * nb);
    return tri_depth(&A, X) > 0.0 && tri_depth(&B, X) > 0.0 && cosang <= cos_min;
}

/* Arguments as sfm_triangulate_tracks, with the track count given directly (n_tracks).  Returns 0, or -1 when the
 * scratch allocation fails. */
int sfm_oracle_triangulate_tracks(int n_images, int S, const int64_t* offsets, const int32_t* obs, int64_t n_tracks, const float* xy,
                                  int xy_stride, const double* cams, const uint8_t* registered, const sfm_triangulate_params* prm,
                                  double* out_X, int32_t* out_ninl, uint8_t* out_status, uint8_t* out_obs_inlier, float* out_obs_error,
                                  int64_t* out_counts)
{
    const double cos_min = cos(prm->min_angle * 0.017453292519943295);     /* computed once, as sfm_triangulate_tracks does */
    const double thr2 = prm->max_error * prm->max_error;
    int64_t longest = 0;
    for (int64_t k = 0; k < n_tracks; ++k)
        if (offsets[k + 1] - offsets[k] > longest) longest = offsets[k + 1] - offsets[k];
    int* cam = (int*)malloc(sizeof(int) * (size_t)(longest + 1));
    double* nx = (double*)malloc(sizeof(double) * (size_t)(longest + 1));
    double* ny = (double*)malloc(sizeof(double) * (size_t)(longest + 1));
    if (!cam || !nx || !ny) {
        free(cam); free(nx); free(ny);
        return -1;
    }
    for (int s = 0; s < 5; ++s) out_counts[s] = 0;
    for (int64_t k = 0; k < n_tracks; ++k) {
        const int64_t o0 = offsets[k];
        const int L = (int)(offsets[k + 1] - o0);
        int bad = 0, M = 0;
        for (int i = 0; i < L; ++i) {
            int img = obs[2 * (o0 + i)], f = obs[2 * (o0 + i) + 1];
            if (img < 0 || img >= n_images || f < 0 || f >= S) { bad = 1; continue; }
            if (registered && !registered[img]) continue;
            const float* p = xy + 2 * ((int64_t)img * xy_stride + f);
            const double* c = cams + 16 * (size_t)img;
            cam[M] = img;
            nx[M] = ((double)p[0] - c[2]) / c[0];
            ny[M] = ((double)p[1] - c[3]) / c[1];
            ++M;
        }
        const tri_track T = {cams, cam, nx, ny, M, thr2};
        int status = 0, cur = 0;
        double X[3] = {0.0, 0.0, 0.0};
        if (bad) {
            status = 4;
        } else if (M < 2) {
            status = 1;
        } else {
            int best = -1, done = 0;
            while (done < prm->max_iters) {
                int nb = ransac_batch(done);
                if (nb > prm->max_iters - done) nb = prm->max_iters - done;
                for (int h = 0; h < nb; ++h) {
                    double Xh[3];
                    if (!tri_hypothesis(&T, prm->seed, (uint32_t)k, done + h, cos_min, Xh)) continue;
                    int n = tri_count(&T, Xh);
                    if (n > best) { best = n; X[0] = Xh[0]; X[1] = Xh[1]; X[2] = Xh[2]; }
                }
                done += nb;
                if (should_stop(best, M, 2, done, prm->confidence)) break;
            }
            if (best < 0) {
                status = 2;
                X[0] = X[1] = X[2] = 0.0;
            } else {
                cur = best;
                for (int round = 0; round < SFM_LO_ROUNDS && cur >= 2; ++round) {
                    double G[10] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, Xr[3];
                    for (int u = 0; u < M; ++u) {
                        tri_camera K;
                        double e2;
                        tri_load_camera(cams + 16 * (size_t)cam[u], &K);
                        if (tri_reproject(&K, X, nx[u], ny[u], thr2, &e2)) tri_add_rows(G, &K, nx[u], ny[u]);
                    }
                    if (!tri_solve(G, Xr)) break;
                    int n = tri_count(&T, Xr);
                    if (n < cur) break;
                    cur = n;
                    X[0] = Xr[0]; X[1] = Xr[1]; X[2] = Xr[2];
                }
                if (cur < prm->min_inliers) {
                    status = 3;
                    X[0] = X[1] = X[2] = 0.0;
                }
            }
        }
        for (int i = 0; i < L; ++i) {
            float err = NAN;
            uint8_t inl = 0;
            if (status == 0) {
                int img = obs[2 * (o0 + i)];
                if (!registered || registered[img]) {
                    const float* p = xy + 2 * ((int64_t)img * xy_stride + obs[2 * (o0 + i) + 1]);
                    const double* c = cams + 16 * (size_t)img;
                    double x = ((double)p[0] - c[2]) / c[0], y = ((double)p[1] - c[3]) / c[1], e2;
                    tri_camera K;
                    tri_load_camera(c, &K);
                    inl = (uint8_t)tri_reproject(&K, X, x, y, thr2, &e2);
                    err = (float)sqrt(e2);
                }
            }
            out_obs_inlier[o0 + i] = inl;
            out_obs_error[o0 + i] = err;
        }
        for (int c = 0; c < 3; ++c) out_X[3 * k + c] = X[c];
        out_ninl[k] = (status == 0 || status == 3) ? cur : 0;
        out_status[k] = (uint8_t)status;
        out_counts[status] += 1;
    }
    free(cam); free(nx); free(ny);
    return 0;
}
