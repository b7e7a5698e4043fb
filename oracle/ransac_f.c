/* ransac_f.c -- CPU oracle for batched RANSAC fundamental-matrix verification.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under sfm-project_b200/ links, imports or
 * executes this file; only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline leg may.
 *
 * What it restates.  The reference's code/geometric_verification.py is a 0-byte
 * file (placeholder comment at code/pipeline.py:60), so there is no reference
 * algorithm to follow line by line.  The conventions (F with x2^T F x1 = 0,
 * F[8] normalised to 1, uint8 mask, inlier iff max(d1^2,d2^2) <= thr^2) are those
 * of cv2.findFundamentalMat(FM_RANSAC) -- OpenCV 4.13.0 (third party, not under
 * /root/reference, version unpinned by the reference) -- as characterised in
 * SURVEY.md Appendix A.4 and pinned by tests/test_oracle_pinned.py against cv2
 * run in this image.  Sampling and termination are this build's own: a
 * counter-based RNG, hypotheses evaluated in batches of 32, 32, 64, then 128 (ransac_batch), and a
 * stop rule that uses only IEEE + - * / sqrt so that the CUDA kernel and this
 * file produce bit-identical masks and counts.  PARITY UNPINNED by the reference
 * (it has no tests); pinned against cv2 statistically (tests/).
 *
 * Build:  gcc -O2 -ffp-contract=off -mfma -fPIC -shared  (oracle/Makefile)
 * Every floating-point operation is written in the order the CUDA kernel
 * (sfm-project_b200/csrc/ransac_f.cu) performs it; no contraction is allowed
 * on either side except the explicit fma()/fmaf() calls.
 */
#include "ransac_common.h"

/* ------------------------------------------------------------ small algebra */
static double det3(const double* r0, const double* r1, const double* r2)
{
    double a = r1[1] * r2[2] - r1[2] * r2[1];
    double b = r1[0] * r2[2] - r1[2] * r2[0];
    double c = r1[0] * r2[1] - r1[1] * r2[0];
    return r0[0] * a - r0[1] * b + r0[2] * c;
}

/* F <- closest rank-2 matrix: remove the component along the right singular
 * vector of the smallest singular value. */
static void enforce_rank2(double* F)
{
    double G[9], V[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            G[i * 3 + j] = F[0 + i] * F[0 + j] + F[3 + i] * F[3 + j] + F[6 + i] * F[6 + j];
    jacobi_eig(G, V, 3, 6);
    int k = 0;
    if (G[4] < G[k * 4]) k = 1;
    if (G[8] < G[k * 4]) k = 2;
    double v0 = V[0 + k], v1 = V[3 + k], v2 = V[6 + k];
    for (int r = 0; r < 3; ++r) {
        double w = F[r * 3 + 0] * v0 + F[r * 3 + 1] * v1 + F[r * 3 + 2] * v2;
        F[r * 3 + 0] -= w * v0;
        F[r * 3 + 1] -= w * v1;
        F[r * 3 + 2] -= w * v2;
    }
}


/* F = T2^T Fh T1, then scale to unit Frobenius norm.  Returns 0 if unusable. */
static int denormalise(const double* Fh, norm2d n1, norm2d n2, double* F)
{
    double G[9];
    for (int r = 0; r < 3; ++r) {
        double f0 = Fh[r * 3 + 0], f1 = Fh[r * 3 + 1], f2 = Fh[r * 3 + 2];
        G[r * 3 + 0] = n1.s * f0;
        G[r * 3 + 1] = n1.s * f1;
        G[r * 3 + 2] = f2 - n1.s * (n1.cx * f0 + n1.cy * f1);
    }
    for (int c = 0; c < 3; ++c) {
        double g0 = G[0 + c], g1 = G[3 + c], g2 = G[6 + c];
        F[0 + c] = n2.s * g0;
        F[3 + c] = n2.s * g1;
        F[6 + c] = g2 - n2.s * (n2.cx * g0 + n2.cy * g1);
    }
    double ss = 0.0;
    for (int i = 0; i < 9; ++i) ss += F[i] * F[i];
    if (!(ss > 0.0) || !(ss < 1e300)) return 0;
    double inv = 1.0 / sqrt(ss);
    for (int i = 0; i < 9; ++i) F[i] *= inv;
    return 1;
}

/* Real roots of c3 x^3 + c2 x^2 + c1 x + c0 using only + - * / sqrt. */
static int solve_cubic(double c3, double c2, double c1, double c0, double* roots)
{
    double mx = fmax(fabs(c2), fmax(fabs(c1), fabs(c0)));
    int n = 0;
    if (!(fabs(c3) > 1e-14 * mx)) {
        /* degenerate: quadratic c2 x^2 + c1 x + c0 */
        if (!(fabs(c2) > 1e-14 * fmax(fabs(c1), fabs(c0)))) {
            if (c1 != 0.0) roots[n++] = -c0 / c1;
            return n;
        }
        double disc = c1 * c1 - 4.0 * c2 * c0;
        if (disc < 0.0) return 0;
        double sq = sqrt(disc);
        double q = -0.5 * (c1 + (c1 >= 0.0 ? sq : -sq));
        roots[n++] = q / c2;
        if (q != 0.0) roots[n++] = c0 / q;
        return n;
    }
    double b = c2 / c3, c = c1 / c3, d = c0 / c3;
    double R = 1.0 + fmax(fabs(b), fmax(fabs(c), fabs(d)));
    double lo = -R, hi = R;
    for (int it = 0; it < 80; ++it) {
        double mid = 0.5 * (lo + hi);
        double fm = ((mid + b) * mid + c) * mid + d;
        if (fm < 0.0) lo = mid; else hi = mid;
    }
    double r = 0.5 * (lo + hi);
    for (int it = 0; it < 2; ++it) {
        double f = ((r + b) * r + c) * r + d;
        double fp = (3.0 * r + 2.0 * b) * r + c;
        if (fp != 0.0) r = r - f / fp;
    }
    roots[n++] = r;
    double B = b + r;
    double C = c + r * B;
    double disc = B * B - 4.0 * C;
    if (disc >= 0.0) {
        double sq = sqrt(disc);
        double q = -0.5 * (B + (B >= 0.0 ? sq : -sq));
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

/* The epipolar row of one normalised correspondence: x2^T F x1 = 0 */
static int rows_f(double u1, double v1, double u2, double v2, double (*r)[9])
{
    r[0][0] = u2 * u1; r[0][1] = u2 * v1; r[0][2] = u2;
    r[0][3] = v2 * u1; r[0][4] = v2 * v1; r[0][5] = v2;
    r[0][6] = u1;      r[0][7] = v1;      r[0][8] = 1.0;
    return 1;
}

/* F from a null vector of the normalised system: the 8-point model, and the LO refit's */
static int refit_f(double* Fh, norm2d n1, norm2d n2, double* F)
{
    enforce_rank2(Fh);
    return denormalise(Fh, n1, n2, F);
}

/* Minimal solver: m = 7 or 8 sample points -> up to 3 unit-norm F (row-major). */
static int solve_minimal(const float* corr, const int* idx, int m, double* Fout)
{
    norm2d n1, n2;
    double N[2][9];
    if (!hartley_null_space(corr, idx, m, rows_f, 1e-12, &n1, &n2, N)) return 0;
    if (m == 8) return refit_f(N[0], n1, n2, Fout);
    /* 7 point: det(l*F1 + F2) = 0 */
    const double* F1 = N[0];
    const double* F2 = N[1];
    double c3 = det3(F1, F1 + 3, F1 + 6);
    double c0 = det3(F2, F2 + 3, F2 + 6);
    double c2 = det3(F2, F1 + 3, F1 + 6) + det3(F1, F2 + 3, F1 + 6) + det3(F1, F1 + 3, F2 + 6);
    double c1 = det3(F1, F2 + 3, F2 + 6) + det3(F2, F1 + 3, F2 + 6) + det3(F2, F2 + 3, F1 + 6);
    double roots[3];
    int nr = solve_cubic(c3, c2, c1, c0, roots);
    int nm = 0;
    for (int r = 0; r < nr; ++r) {
        double Fh[9];
        for (int i = 0; i < 9; ++i) Fh[i] = roots[r] * F1[i] + F2[i];
        if (denormalise(Fh, n1, n2, Fout + 9 * nm)) ++nm;
    }
    return nm;
}

/* ------------------------------------------------------------------ scoring */
static int is_inlier(const float* Ff, const float* c, float thr2, int score)
{
    float x1 = c[0], y1 = c[1], x2 = c[2], y2 = c[3];
    float a = fmaf(Ff[0], x1, fmaf(Ff[1], y1, Ff[2]));
    float b = fmaf(Ff[3], x1, fmaf(Ff[4], y1, Ff[5]));
    float cc = fmaf(Ff[6], x1, fmaf(Ff[7], y1, Ff[8]));
    float num = fmaf(x2, a, fmaf(y2, b, cc));
    float a2 = fmaf(Ff[0], x2, fmaf(Ff[3], y2, Ff[6]));
    float b2 = fmaf(Ff[1], x2, fmaf(Ff[4], y2, Ff[7]));
    float bb = b * b;
    float s1 = fmaf(a, a, bb);
    float bb2 = b2 * b2;
    float s2 = fmaf(a2, a2, bb2);
    float n2 = num * num;
    float lim = (score == SFM_SCORE_SAMPSON) ? thr2 * (s1 + s2) : thr2 * fminf(s1, s2);
    return n2 <= lim;
}

/* --------------------------------------------------------------- driver */
static int sample_size_f(const sfm_ransac_params* prm) { return (prm->solver == 7 || prm->solver == 8) ? prm->solver : 0; }

/* LO needs 8 inliers for the 7-point solver too */
static const oracle_model kFundamental = {sample_size_f, solve_minimal, is_inlier, rows_f, 8, refit_f};

int sfm_oracle_ransac_f(const float* corr, int M, const sfm_ransac_params* prm, uint32_t pair_id,
                        const uint32_t* samples, double* out_F, int32_t* out_ninl,
                        uint8_t* out_mask, int32_t* out_iters)
{
    return oracle_ransac_driver(&kFundamental, corr, M, prm, pair_id, samples, 0, out_F, out_ninl, out_mask, out_iters);
}

/* Expose the pieces so tests can pin them individually. */
int sfm_oracle_solve_minimal(const float* corr, const int32_t* idx, int m, double* Fout)
{
    int id[8];
    for (int k = 0; k < m; ++k) id[k] = idx[k];
    return solve_minimal(corr, id, m, Fout);
}

int sfm_oracle_count_inliers(const double* F, const float* corr, int M, float thr, int score, uint8_t* mask)
{
    return count_inliers(is_inlier, F, corr, M, thr * thr, score, mask);
}

void sfm_oracle_draw_sample(uint64_t seed, uint32_t pair, uint32_t hyp, int m, int M, int32_t* idx)
{
    int id[8];
    draw_sample(seed, pair, hyp, m, M, id);
    for (int k = 0; k < m; ++k) idx[k] = id[k];
}

int sfm_oracle_smallest_eigvec9(const double* A, double* x) { return smallest_eigvec9(A, x); }
