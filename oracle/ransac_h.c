/* ransac_h.c -- CPU oracle for batched RANSAC homography estimation.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under sfm-project_b200/ links, imports or
 * executes this file; only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline leg may.
 *
 * What it restates.  The reference's code/geometric_verification.py is a 0-byte
 * file (placeholder at code/pipeline.py:60-65); SURVEY.md section 8f rank 2 asks
 * for the homography model beside F.  Conventions (x2 ~ H x1, H[8] normalised to
 * 1, uint8 mask, inlier iff |proj(H x1) - x2|^2 <= thr^2) are those of
 * cv2.findHomography(RANSAC) -- OpenCV 4.13.0, third party, unpinned by the
 * reference -- pinned statistically by tests/test_oracle_pinned.py against cv2
 * run in this image.  Sampling / termination are this build's own seeded scheme
 * (the same as ransac_f.c).  PARITY UNPINNED by the reference (it has no tests).
 *
 * Operation for operation the same as sfm-project_b200/csrc/ransac_h.cu; built
 * with -ffp-contract=off so masks, counts and H are compared bit for bit.
 */
#include "ransac_common.h"

static int denormalise_h(const double* Hn, norm2d n1, norm2d n2, double* H)
{
    double G[9];
    for (int r = 0; r < 3; ++r) {
        double h0 = Hn[r * 3 + 0], h1 = Hn[r * 3 + 1], h2 = Hn[r * 3 + 2];
        G[r * 3 + 0] = n1.s * h0;
        G[r * 3 + 1] = n1.s * h1;
        G[r * 3 + 2] = h2 - n1.s * (n1.cx * h0 + n1.cy * h1);
    }
    double is2 = 1.0 / n2.s;
    for (int c = 0; c < 3; ++c) {
        double g0 = G[0 + c], g1 = G[3 + c], g2 = G[6 + c];
        H[0 + c] = is2 * g0 + n2.cx * g2;
        H[3 + c] = is2 * g1 + n2.cy * g2;
        H[6 + c] = g2;
    }
    double ss = 0.0;
    for (int i = 0; i < 9; ++i) ss += H[i] * H[i];
    if (!(ss > 0.0) || !(ss < 1e300)) return 0;
    double inv = 1.0 / sqrt(ss);
    for (int i = 0; i < 9; ++i) H[i] *= inv;
    return 1;
}

/* The two DLT rows of one normalised correspondence: x2 ~ H x1 */
static int rows_h(double u1, double v1, double u2, double v2, double (*r)[9])
{
    double* r0 = r[0];
    double* r1 = r[1];
    r0[0] = u1;  r0[1] = v1;  r0[2] = 1.0; r0[3] = 0.0; r0[4] = 0.0; r0[5] = 0.0;
    r0[6] = -(u2 * u1); r0[7] = -(u2 * v1); r0[8] = -u2;
    r1[0] = 0.0; r1[1] = 0.0; r1[2] = 0.0; r1[3] = u1;  r1[4] = v1;  r1[5] = 1.0;
    r1[6] = -(v2 * u1); r1[7] = -(v2 * v1); r1[8] = -v2;
    return 2;
}

static int solve_h4(const float* corr, const int* idx, int m, double* Hout)
{
    norm2d n1, n2;
    double N[2][9];
    if (!hartley_null_space(corr, idx, 4, rows_h, 1e-10, &n1, &n2, N)) return 0;
    if (!denormalise_h(N[0], n1, n2, Hout)) return 0;
    /* the sample points map with w of one sign */
    int pos = 0, neg = 0;
    for (int k = 0; k < 4; ++k) {
        const float* c = corr + 4 * (size_t)idx[k];
        double w = Hout[6] * (double)c[0] + Hout[7] * (double)c[1] + Hout[8];
        pos += (w > 0.0);
        neg += (w < 0.0);
    }
    return (pos == 4 || neg == 4) ? 1 : 0;
}

static int is_inlier_h(const float* H, const float* c, float thr2, int score)
{
    float X = fmaf(H[0], c[0], fmaf(H[1], c[1], H[2]));
    float Y = fmaf(H[3], c[0], fmaf(H[4], c[1], H[5]));
    float W = fmaf(H[6], c[0], fmaf(H[7], c[1], H[8]));
    float ex = fmaf(-c[2], W, X);
    float ey = fmaf(-c[3], W, Y);
    float ey2 = ey * ey;
    float e2 = fmaf(ex, ex, ey2);
    float lim = thr2 * (W * W);
    return e2 <= lim && lim > 0.f;
}

static int refit_h(double* Hn, norm2d n1, norm2d n2, double* H) { return denormalise_h(Hn, n1, n2, H); }

static int sample_size_h(const sfm_ransac_params* prm) { return 4; }

static const oracle_model kHomography = {sample_size_h, solve_h4, is_inlier_h, rows_h, 4, refit_h};

int sfm_oracle_ransac_h(const float* corr, int M, const sfm_ransac_params* prm, uint32_t pair_id,
                        const uint32_t* samples, int stop_target, double* out_H, int32_t* out_ninl,
                        uint8_t* out_mask, int32_t* out_iters)
{
    return oracle_ransac_driver(&kHomography, corr, M, prm, pair_id, samples, stop_target, out_H, out_ninl, out_mask, out_iters);
}

int sfm_oracle_solve_h4(const float* corr, const int32_t* idx, double* Hout)
{
    int id[4];
    for (int k = 0; k < 4; ++k) id[k] = idx[k];
    return solve_h4(corr, id, 4, Hout);
}

int sfm_oracle_count_inliers_h(const double* H, const float* corr, int M, float thr, uint8_t* mask)
{
    return count_inliers(is_inlier_h, H, corr, M, thr * thr, 0, mask);
}
