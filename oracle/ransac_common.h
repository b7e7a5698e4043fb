/* ransac_common.h -- helpers shared by the CPU oracles (ransac_f.c, ransac_h.c, pose.c), and the RANSAC driver that
 * runs RANSAC-F and RANSAC-H.  Each of those two supplies only an oracle_model (see below), as the kernels supply a
 * Model policy to ransac_driver.
 *
 * TEST INFRASTRUCTURE ONLY (see ransac_f.c).  Operation for operation the same as
 * sfm-project_b200/csrc/ransac_common.cuh; built with -ffp-contract=off.
 */
#ifndef SFM_ORACLE_RANSAC_COMMON_H
#define SFM_ORACLE_RANSAC_COMMON_H
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../include/sfm_b200.h"

/* hypotheses evaluated before the next termination check: 32, 32, 64, then 128 at a time */
static __attribute__((unused)) int ransac_batch(int done) { return done < 64 ? 32 : (done < 128 ? 64 : 128); }
#define SFM_RANSAC_LANES 256      /* virtual reduction lanes of the LO refit    */
#define SFM_LO_ROUNDS 2

typedef struct { double s, cx, cy; } norm2d;

/* ---------------------------------------------------------------- sampling */
static __attribute__((unused)) uint32_t rng_u32(uint64_t seed, uint32_t pair, uint32_t hyp, uint32_t ctr)
{
    uint64_t x = seed + 0x9E3779B97F4A7C15ULL * ((((uint64_t)pair) << 32) | (uint64_t)hyp);
    x ^= 0xD1B54A32D192ED03ULL * (uint64_t)(ctr + 1u);
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ULL;
    x ^= x >> 27; x *= 0x94D049BB133111EBULL;
    x ^= x >> 31;
    return (uint32_t)(x >> 32);
}

static __attribute__((unused)) void draw_sample(uint64_t seed, uint32_t pair, uint32_t hyp, int m, int M, int* idx)
{
    for (int k = 0; k < m; ++k) {
        int v = 0;
        for (int attempt = 0; attempt < 16; ++attempt) {
            uint32_t r = rng_u32(seed, pair, hyp, (uint32_t)(k * 16 + attempt));
            v = (int)(((uint64_t)r * (uint64_t)(uint32_t)M) >> 32);
            int dup = 0;
            for (int j = 0; j < k; ++j) dup |= (idx[j] == v);
            if (!dup) break;
        }
        idx[k] = v;
    }
}

/* The m correspondence indices of hypothesis hyp: the caller's samples rows ([max_iters, 8], reduced mod M) or drawn.
 * Kernel twin: hypothesis_sample. */
static __attribute__((unused)) void hypothesis_sample(const uint32_t* samples, uint64_t seed, uint32_t pair, int hyp, int m,
                                                      int M, int* idx)
{
    if (samples) {
        for (int k = 0; k < m; ++k) idx[k] = (int)(samples[(size_t)hyp * 8 + k] % (uint32_t)M);
    } else {
        draw_sample(seed, pair, (uint32_t)hyp, m, M, idx);
    }
}

/* cyclic Jacobi eigen-decomposition of a symmetric n x n matrix (n <= 9).
 * A is destroyed (diagonal = eigenvalues), V gets eigenvectors in columns. */
static __attribute__((unused)) void jacobi_eig(double* A, double* V, int n, int sweeps)
{
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) V[i * n + j] = (i == j) ? 1.0 : 0.0;
    for (int s = 0; s < sweeps; ++s) {
        for (int p = 0; p < n - 1; ++p) {
            for (int q = p + 1; q < n; ++q) {
                double apq = A[p * n + q];
                if (apq == 0.0) continue;
                double app = A[p * n + p], aqq = A[q * n + q];
                double theta = (aqq - app) / (2.0 * apq);
                double at = fabs(theta);
                double t = 1.0 / (at + sqrt(theta * theta + 1.0));
                if (theta < 0.0) t = -t;
                double c = 1.0 / sqrt(t * t + 1.0);
                double sn = t * c;
                for (int k = 0; k < n; ++k) {        /* columns p,q */
                    double akp = A[k * n + p], akq = A[k * n + q];
                    A[k * n + p] = c * akp - sn * akq;
                    A[k * n + q] = sn * akp + c * akq;
                }
                for (int k = 0; k < n; ++k) {        /* rows p,q */
                    double apk = A[p * n + k], aqk = A[q * n + k];
                    A[p * n + k] = c * apk - sn * aqk;
                    A[q * n + k] = sn * apk + c * aqk;
                }
                for (int k = 0; k < n; ++k) {
                    double vkp = V[k * n + p], vkq = V[k * n + q];
                    V[k * n + p] = c * vkp - sn * vkq;
                    V[k * n + q] = sn * vkp + c * vkq;
                }
            }
        }
    }
}

/* stop when (1 - w^m)^done <= 1 - confidence, IEEE basic ops only */
static __attribute__((unused)) int should_stop(int best, int M, int m, int done, double confidence)
{
    if (confidence >= 1.0 || best <= 0) return 0;
    double w = (double)best / (double)M;
    double wm = 1.0;
    for (int k = 0; k < m; ++k) wm *= w;
    double q = 1.0 - wm;
    if (!(q > 0.0)) return 1;
    double res = 1.0, base = q;
    int e = done;
    while (e) { if (e & 1) res *= base; base *= base; e >>= 1; }
    return res <= (1.0 - confidence);
}

static __attribute__((unused)) double lane_tree(double* v /* [SFM_RANSAC_LANES] partials */)
{
    /* per 32-lane warp: shfl_down tree; then warps summed in order */
    double total = 0.0;
    for (int w = 0; w < SFM_RANSAC_LANES / 32; ++w) {
        double* l = v + 32 * w;
        for (int off = 16; off >= 1; off >>= 1)
            for (int i = 0; i < off; ++i) l[i] += l[i + off];
        total = (w == 0) ? l[0] : total + l[0];
    }
    return total;
}


/* Eigenvector of the smallest eigenvalue of a symmetric positive semi-definite 9 x 9 matrix: Cholesky factor of
 * A + eps*I (eps = 1e-13 * trace), then inverse iterations from a fixed start vector until the normalised iterate stops
 * moving (at most 16).  Operation for operation
 * smallest_eigvec9 of csrc/ransac_common.cuh. */
static __attribute__((unused)) int smallest_eigvec9(const double* A, double* xout)
{
    double L[45], invd[9], x[9], y[9], z[9];
    double tr = 0.0;
    for (int i = 0; i < 9; ++i) tr += A[i * 9 + i];
    if (!(tr > 0.0) || !(tr < 1e300)) return 0;
    const double eps = tr * 1e-13;
    for (int j = 0; j < 9; ++j) {
        double sj = A[j * 9 + j] + eps;
        for (int k = 0; k < j; ++k) sj -= L[j * (j + 1) / 2 + k] * L[j * (j + 1) / 2 + k];
        if (!(sj > 0.0)) return 0;
        const double d = sqrt(sj);
        L[j * (j + 1) / 2 + j] = d;
        invd[j] = 1.0 / d;
        for (int i = j + 1; i < 9; ++i) {
            double v = A[i * 9 + j];
            for (int k = 0; k < j; ++k) v -= L[i * (i + 1) / 2 + k] * L[j * (j + 1) / 2 + k];
            L[i * (i + 1) / 2 + j] = v * invd[j];
        }
    }
    for (int i = 0; i < 9; ++i) x[i] = 1.0 + 0.125 * (double)i;
    for (int it = 0; it < 16; ++it) {
        for (int i = 0; i < 9; ++i) {
            double v = x[i];
            for (int k = 0; k < i; ++k) v -= L[i * (i + 1) / 2 + k] * y[k];
            y[i] = v * invd[i];
        }
        for (int i = 8; i >= 0; --i) {
            double v = y[i];
            for (int k = i + 1; k < 9; ++k) v -= L[k * (k + 1) / 2 + i] * z[k];
            z[i] = v * invd[i];
        }
        double ss = 0.0;
        for (int i = 0; i < 9; ++i) ss += z[i] * z[i];
        if (!(ss > 0.0) || !(ss < 1e300)) return 0;
        const double inv = 1.0 / sqrt(ss);
        double diff = 0.0;
        for (int i = 0; i < 9; ++i) {
            const double xi = z[i] * inv;
            diff = fmax(diff, fabs(xi - x[i]));
            x[i] = xi;
        }
        if (it > 0 && diff < 1e-13) break;
    }
    for (int i = 0; i < 9; ++i) xout[i] = x[i];
    return 1;
}

/* ------------------------------------------------------------ the RANSAC driver */
/* The rows (1 or 2) that one Hartley-normalised correspondence adds to a model's linear system, in the minimal solver
 * and in the LO refit */
typedef int (*model_rows_fn)(double u1, double v1, double u2, double v2, double (*r)[9]);
/* fp32 inlier predicate of a model rounded to float */
typedef int (*inlier_fn)(const float* model, const float* c, float thr2, int score);

/* What RANSAC-F and RANSAC-H supply to oracle_ransac_driver; the kernel twin is the Model policy of ransac_driver. */
typedef struct {
    int (*sample_size)(const sfm_ransac_params* prm);              /* m; 0 when prm names no solver of this model */
    int (*solve)(const float* corr, const int* idx, int m, double* out);   /* up to 3 unit-norm models; returns their number */
    inlier_fn inlier;
    model_rows_fn rows;
    int lo_min;                                                    /* fewest inliers the LO refit runs on */
    int (*refit)(double* h, norm2d n1, norm2d n2, double* out);    /* model from the smallest eigenvector h; 0 if unusable */
} oracle_model;

/* Hartley normalisation (n1, n2) of the m-point sample idx, then the null space of the n rows (at most 8) that `rows`
 * makes from its points, by Gauss-Jordan elimination with complete pivoting: 9 - n vectors in N.  Returns 9 - n; 0 when
 * the points of either image coincide or a pivot is not above tol.  Kernel twins: hartley_sample and coop_gauss_jordan. */
static __attribute__((unused)) int hartley_null_space(const float* corr, const int* idx, int m, model_rows_fn rows, double tol,
                                                      norm2d* n1, norm2d* n2, double N[2][9])
{
    double x1[8], y1[8], x2[8], y2[8];
    for (int k = 0; k < m; ++k) {
        const float* c = corr + 4 * (size_t)idx[k];
        x1[k] = (double)c[0]; y1[k] = (double)c[1];
        x2[k] = (double)c[2]; y2[k] = (double)c[3];
    }
    {
        double sx = 0.0, sy = 0.0, tx = 0.0, ty = 0.0;
        for (int k = 0; k < m; ++k) { sx += x1[k]; sy += y1[k]; tx += x2[k]; ty += y2[k]; }
        double inv = 1.0 / (double)m;
        n1->cx = sx * inv; n1->cy = sy * inv; n2->cx = tx * inv; n2->cy = ty * inv;
        double d1 = 0.0, d2 = 0.0;
        for (int k = 0; k < m; ++k) {
            double ax = x1[k] - n1->cx, ay = y1[k] - n1->cy;
            double bx = x2[k] - n2->cx, by = y2[k] - n2->cy;
            d1 += sqrt(ax * ax + ay * ay);
            d2 += sqrt(bx * bx + by * by);
        }
        d1 *= inv; d2 *= inv;
        if (!(d1 > 1e-9) || !(d2 > 1e-9)) return 0;
        n1->s = 1.4142135623730951 / d1;
        n2->s = 1.4142135623730951 / d2;
    }
    double A[8][9];
    int n = 0;
    for (int k = 0; k < m; ++k) {
        double u1 = (x1[k] - n1->cx) * n1->s, v1 = (y1[k] - n1->cy) * n1->s;
        double u2 = (x2[k] - n2->cx) * n2->s, v2 = (y2[k] - n2->cy) * n2->s;
        n += rows(u1, v1, u2, v2, A + n);
    }
    int perm[9];
    for (int j = 0; j < 9; ++j) perm[j] = j;
    for (int k = 0; k < n; ++k) {
        int pi = k, pj = k;
        double best = -1.0;
        for (int i = k; i < n; ++i)
            for (int j = k; j < 9; ++j) {
                double v = fabs(A[i][j]);
                if (v > best) { best = v; pi = i; pj = j; }
            }
        if (!(best > tol)) return 0;
        if (pi != k)
            for (int j = 0; j < 9; ++j) { double t = A[k][j]; A[k][j] = A[pi][j]; A[pi][j] = t; }
        if (pj != k) {
            for (int i = 0; i < n; ++i) { double t = A[i][k]; A[i][k] = A[i][pj]; A[i][pj] = t; }
            int t = perm[k]; perm[k] = perm[pj]; perm[pj] = t;
        }
        double inv = 1.0 / A[k][k];
        for (int j = k; j < 9; ++j) A[k][j] *= inv;
        for (int i = 0; i < n; ++i) {
            if (i == k) continue;
            double f = A[i][k];
            for (int j = k; j < 9; ++j) A[i][j] -= f * A[k][j];
        }
    }
    for (int c = 0; c < 9 - n; ++c) {
        for (int j = 0; j < 9; ++j) N[c][j] = 0.0;
        N[c][perm[n + c]] = 1.0;
        for (int k = 0; k < n; ++k) N[c][perm[k]] = -A[k][n + c];
    }
    return 9 - n;
}

/* Inliers of a model after rounding it to float; mask may be NULL.  Kernel twin: block_count_inliers. */
static __attribute__((unused)) int count_inliers(inlier_fn inlier, const double* model, const float* corr, int M, float thr2,
                                                 int score, uint8_t* mask)
{
    float Mf[9];
    for (int i = 0; i < 9; ++i) Mf[i] = (float)model[i];
    int n = 0;
    for (int i = 0; i < M; ++i) {
        int in = inlier(Mf, corr + 4 * (size_t)i, thr2, score);
        if (mask) mask[i] = (uint8_t)in;
        n += in;
    }
    return n;
}

/* LO: Hartley-normalised least-squares refit on the inliers in mask -- moments, mean distances and the 9 x 9 normal
 * matrix of the model's rows, each summed over SFM_RANSAC_LANES lanes and lane_tree, then its smallest eigenvector.
 * Kernel twin: the LO step of ransac_driver. */
static __attribute__((unused)) int lo_refit(const oracle_model* mdl, const float* corr, int M, const uint8_t* mask, double* out)
{
    double part[SFM_RANSAC_LANES];
    double mom[5];
    for (int q = 0; q < 5; ++q) {
        for (int t = 0; t < SFM_RANSAC_LANES; ++t) {
            double s = 0.0;
            for (int i = t; i < M; i += SFM_RANSAC_LANES)
                if (mask[i]) s += (q == 4) ? 1.0 : (double)corr[4 * (size_t)i + q];
            part[t] = s;
        }
        mom[q] = lane_tree(part);
    }
    if (!(mom[4] >= (double)mdl->lo_min)) return 0;
    norm2d n1, n2;
    double inv = 1.0 / mom[4];
    n1.cx = mom[0] * inv; n1.cy = mom[1] * inv; n2.cx = mom[2] * inv; n2.cy = mom[3] * inv;
    double dd[2];
    for (int q = 0; q < 2; ++q) {
        double cx = q ? n2.cx : n1.cx, cy = q ? n2.cy : n1.cy;
        for (int t = 0; t < SFM_RANSAC_LANES; ++t) {
            double s = 0.0;
            for (int i = t; i < M; i += SFM_RANSAC_LANES)
                if (mask[i]) {
                    double ax = (double)corr[4 * (size_t)i + 2 * q] - cx;
                    double ay = (double)corr[4 * (size_t)i + 2 * q + 1] - cy;
                    s += sqrt(ax * ax + ay * ay);
                }
            part[t] = s;
        }
        dd[q] = lane_tree(part) * inv;
    }
    if (!(dd[0] > 1e-9) || !(dd[1] > 1e-9)) return 0;
    n1.s = 1.4142135623730951 / dd[0];
    n2.s = 1.4142135623730951 / dd[1];
    double AtA[81];
    for (int a = 0; a < 9; ++a)
        for (int b = a; b < 9; ++b) {
            for (int t = 0; t < SFM_RANSAC_LANES; ++t) {
                double s = 0.0;
                for (int i = t; i < M; i += SFM_RANSAC_LANES)
                    if (mask[i]) {
                        const float* c = corr + 4 * (size_t)i;
                        double u1 = ((double)c[0] - n1.cx) * n1.s, v1 = ((double)c[1] - n1.cy) * n1.s;
                        double u2 = ((double)c[2] - n2.cx) * n2.s, v2 = ((double)c[3] - n2.cy) * n2.s;
                        double r[2][9];
                        int nr = mdl->rows(u1, v1, u2, v2, r);
                        for (int j = 0; j < nr; ++j) s += r[j][a] * r[j][b];
                    }
                part[t] = s;
            }
            double v = lane_tree(part);
            AtA[a * 9 + b] = v;
            AtA[b * 9 + a] = v;
        }
    double h[9];
    if (!smallest_eigvec9(AtA, h)) return 0;
    return mdl->refit(h, n1, n2, out);
}

/* One RANSAC run on the M correspondences corr (x1, y1, x2, y2): hypotheses in batches of ransac_batch, strict-greater
 * selection in (hypothesis, root) order, the stop rule on max(best, stop_target clamped to [0, M]), the final mask, the
 * LO rounds and the min_inliers rule.  out_mask and out_iters may be NULL.  The model is divided by its element [8]
 * (cv2's convention).  Kernel twin: ransac_driver. */
static __attribute__((unused)) int oracle_ransac_driver(const oracle_model* mdl, const float* corr, int M,
                                                        const sfm_ransac_params* prm, uint32_t pair_id, const uint32_t* samples,
                                                        int stop_target, double* out_model, int32_t* out_ninl,
                                                        uint8_t* out_mask, int32_t* out_iters)
{
    const int m = mdl->sample_size(prm);
    const float thr2 = prm->threshold * prm->threshold;
    for (int i = 0; i < 9; ++i) out_model[i] = 0.0;
    if (out_mask) memset(out_mask, 0, (size_t)(M > 0 ? M : 0));
    *out_ninl = 0;
    if (out_iters) *out_iters = 0;
    if (m == 0 || M < m) return 0;

    double bestM[9];
    int best = 0, done = 0;
    while (done < prm->max_iters) {
        int nb = prm->max_iters - done;
        if (nb > ransac_batch(done)) nb = ransac_batch(done);
        for (int h = 0; h < nb; ++h) {
            int idx[8];
            hypothesis_sample(samples, prm->seed, pair_id, done + h, m, M, idx);
            double Mm[27];
            int nm = mdl->solve(corr, idx, m, Mm);
            for (int r = 0; r < nm; ++r) {
                int cnt = count_inliers(mdl->inlier, Mm + 9 * r, corr, M, thr2, prm->score, NULL);
                if (cnt > best) { best = cnt; memcpy(bestM, Mm + 9 * r, sizeof bestM); }
            }
        }
        done += nb;
        int target = stop_target < 0 ? 0 : (stop_target > M ? M : stop_target);
        if (should_stop(best > target ? best : target, M, m, done, prm->confidence)) break;
    }
    if (out_iters) *out_iters = done;
    if (best < m) return 0;

    uint8_t* mask = out_mask ? out_mask : (uint8_t*)malloc((size_t)M);
    best = count_inliers(mdl->inlier, bestM, corr, M, thr2, prm->score, mask);
    if (prm->lo_refit) {
        uint8_t* trial = (uint8_t*)malloc((size_t)M);
        for (int round = 0; round < SFM_LO_ROUNDS; ++round) {
            double Mr[9];
            if (!lo_refit(mdl, corr, M, mask, Mr)) break;
            int cnt = count_inliers(mdl->inlier, Mr, corr, M, thr2, prm->score, trial);
            if (cnt <= best) break;
            best = cnt;
            memcpy(bestM, Mr, sizeof bestM);
            memcpy(mask, trial, (size_t)M);
        }
        free(trial);
    }
    if (prm->min_inliers > 0 && best < prm->min_inliers) {
        memset(mask, 0, (size_t)M);
        if (!out_mask) free(mask);
        return 0;
    }
    if (!out_mask) free(mask);
    /* cv2 convention model[2,2] == 1.0 exactly: divide (x / x == 1), never multiply by a reciprocal */
    const double s = (fabs(bestM[8]) > 1.1920928955078125e-07) ? bestM[8] : 1.0;
    for (int i = 0; i < 9; ++i) out_model[i] = bestM[i] / s;
    *out_ninl = best;
    return 0;
}
#endif
