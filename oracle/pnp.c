/* pnp.c -- CPU oracle for registration by RANSAC-PnP (sfm_pnp_ransac).
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under sfm-project_b200/ links, imports or executes this file; only tests/ and
 * tools/ may.
 *
 * What it restates: the contract of include/sfm_b200.h, "absolute pose / registration", serially -- one query after
 * another, hypotheses in index order and their poses in root order (strict-greater selection, as the kernel's in-order
 * argmax), the refinement's sums over 256 virtual lanes reduced by lane_tree (the kernel's block_tree_sum_many).  Operation
 * for operation the same as sfm-project_b200/csrc/pnp.cu; built with -ffp-contract=off so poses, counts, statuses and masks
 * are compared bit for bit.  Sampling, the stop rule, the Jacobi solver and lane_tree come from ransac_common.h.
 */
#include "ransac_common.h"

#define PNP_SUMS 28

typedef struct {
    double fx, fy, r[9], t[3];
} pnp_camera;

static int pnp_finite(double v) { return fabs(v) <= 1.7976931348623157e308; }

/* track triangulation's predicate (triangulate.c's tri_reproject) */
static int pnp_reproject(const pnp_camera* K, const double* X, double x, double y, double thr2, double* e2)
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

/* ---------------------------------------------------------------- Lambda Twist P3P (kernel twin: p3p and helpers) */
static double p3p_cubic(double b, double c, double d)
{
    double r0;
    if (b * b >= 3.0 * c) {
        double v = sqrt(b * b - 3.0 * c);
        double t1 = (-b - v) / 3.0;
        double k = ((t1 + b) * t1 + c) * t1 + d;
        if (k > 0.0) {
            r0 = t1 - sqrt(-k / (3.0 * t1 + b));
        } else {
            double t2 = (-b + v) / 3.0;
            k = ((t2 + b) * t2 + c) * t2 + d;
            r0 = t2 + sqrt(-k / (3.0 * t2 + b));
        }
    } else {
        r0 = -b / 3.0;
        if (fabs((3.0 * r0 + 2.0 * b) * r0 + c) < 1e-4) r0 = r0 + 1.0;
    }
    for (int it = 0; it < 50; ++it) {
        double fx = ((r0 + b) * r0 + c) * r0 + d;
        if (!(it < 7 || fabs(fx) > 1e-13)) break;
        double fpx = (3.0 * r0 + 2.0 * b) * r0 + c;
        r0 = r0 - fx / fpx;
    }
    return r0;
}

static void p3p_refine_depths(double L[3], double a12, double a13, double a23, double b12, double b13, double b23)
{
    for (int it = 0; it < 5; ++it) {
        double l1 = L[0], l2 = L[1], l3 = L[2];
        double r1 = l1 * l1 + l2 * l2 + b12 * l1 * l2 - a12;
        double r2 = l1 * l1 + l3 * l3 + b13 * l1 * l3 - a13;
        double r3 = l2 * l2 + l3 * l3 + b23 * l2 * l3 - a23;
        double rs = fabs(r1) + fabs(r2) + fabs(r3);
        if (rs < 1e-10) break;
        double v0 = 2.0 * l1 + b12 * l2, v1 = 2.0 * l2 + b12 * l1;
        double v3 = 2.0 * l1 + b13 * l3, v5 = 2.0 * l3 + b13 * l1;
        double v7 = 2.0 * l2 + b23 * l3, v8 = 2.0 * l3 + b23 * l2;
        double det = 1.0 / (-v0 * v5 * v7 - v1 * v3 * v8);
        double n1 = l1 - det * (-v5 * v7 * r1 + -v1 * v8 * r2 + v1 * v5 * r3);
        double n2 = l2 - det * (-v3 * v8 * r1 + v0 * v8 * r2 + -v0 * v5 * r3);
        double n3 = l3 - det * (v3 * v7 * r1 + -v0 * v7 * r2 + -v1 * v3 * r3);
        double s1 = n1 * n1 + n2 * n2 + b12 * n1 * n2 - a12;
        double s2 = n1 * n1 + n3 * n3 + b13 * n1 * n3 - a13;
        double s3 = n2 * n2 + n3 * n3 + b23 * n2 * n3 - a23;
        if (fabs(s1) + fabs(s2) + fabs(s3) > rs) break;
        L[0] = n1; L[1] = n2; L[2] = n3;
    }
}

static void p3p_line(double s, const double V[9], int e0, int e1, double a12, double a13, double a23, double b12, double b13,
                     double b23, double Ls[4][3], int* n)
{
    double w2 = 1.0 / (s * V[e1] - V[e0]);
    double w0 = (V[3 + e0] - s * V[3 + e1]) * w2;
    double w1 = (V[6 + e0] - s * V[6 + e1]) * w2;
    double a = 1.0 / ((a13 - a12) * w1 * w1 - a12 * b13 * w1 - a12);
    double b = (a13 * b12 * w1 - a12 * b13 * w0 - 2.0 * w0 * w1 * (a12 - a13)) * a;
    double c = ((a13 - a12) * w0 * w0 + a13 * b12 * w0 + a13) * a;
    double disc = b * b - 4.0 * c;
    if (!(disc >= 0.0)) return;
    double y = sqrt(disc);
    double tau1 = b < 0.0 ? 0.5 * (-b + y) : 0.5 * (-b - y);
    double tau2 = c / tau1;
    for (int k = 0; k < 2; ++k) {
        double tau = k == 0 ? tau1 : tau2;
        if (!(tau > 0.0)) continue;
        double d = a23 / (tau * (b23 + tau) + 1.0);
        if (!(d > 0.0)) continue;
        double l2 = sqrt(d);
        double l3 = tau * l2;
        double l1 = w0 * l2 + w1 * l3;
        if (!(l1 >= 0.0)) continue;
        Ls[*n & 3][0] = l1; Ls[*n & 3][1] = l2; Ls[*n & 3][2] = l3;
        *n = *n + 1;
    }
}

/* Up to 4 poses (R row-major, t) of three normalised observations (nx, ny) and world points X (row k = point k). */
int sfm_oracle_p3p(const double nx[3], const double ny[3], const double X[9], double* out)
{
    double y[3][3];
    for (int k = 0; k < 3; ++k) {
        double inv = 1.0 / sqrt(nx[k] * nx[k] + ny[k] * ny[k] + 1.0);
        y[k][0] = nx[k] * inv; y[k][1] = ny[k] * inv; y[k][2] = inv;
    }
    double b12 = -2.0 * (y[0][0] * y[1][0] + y[0][1] * y[1][1] + y[0][2] * y[1][2]);
    double b13 = -2.0 * (y[0][0] * y[2][0] + y[0][1] * y[2][1] + y[0][2] * y[2][2]);
    double b23 = -2.0 * (y[1][0] * y[2][0] + y[1][1] * y[2][1] + y[1][2] * y[2][2]);
    double d12[3], d13[3], d23[3];
    for (int c = 0; c < 3; ++c) {
        d12[c] = X[c] - X[3 + c];
        d13[c] = X[c] - X[6 + c];
        d23[c] = X[3 + c] - X[6 + c];
    }
    double a12 = d12[0] * d12[0] + d12[1] * d12[1] + d12[2] * d12[2];
    double a13 = d13[0] * d13[0] + d13[1] * d13[1] + d13[2] * d13[2];
    double a23 = d23[0] * d23[0] + d23[1] * d23[1] + d23[2] * d23[2];
    double c31 = -0.5 * b13, c23 = -0.5 * b23, c12 = -0.5 * b12;
    double blob = c12 * c23 * c31 - 1.0;
    double s31 = 1.0 - c31 * c31, s23 = 1.0 - c23 * c23, s12 = 1.0 - c12 * c12;
    double p3 = a13 * (a23 * s31 - a13 * s23);
    double p2 = 2.0 * blob * a23 * a13 + a13 * (2.0 * a12 + a13) * s23 + a23 * (a23 - a12) * s31;
    double p1 = a23 * (a13 - a23) * s12 - a12 * a12 * s23 - 2.0 * a12 * (blob * a23 + a13 * s23);
    double p0 = a12 * (a12 * s23 - a23 * s12);
    p3 = 1.0 / p3;
    p2 = p2 * p3; p1 = p1 * p3; p0 = p0 * p3;
    double g = p3p_cubic(p2, p1, p0);
    double A[9], V[9];
    A[0] = a23 * (1.0 - g);
    A[1] = (a23 * b12) * 0.5;
    A[2] = (a23 * b13 * g) * (-0.5);
    A[4] = a23 - a12 + a13 * g;
    A[5] = b23 * (a13 * g - a12) * 0.5;
    A[8] = g * (a13 - a23) - a12;
    A[3] = A[1]; A[6] = A[2]; A[7] = A[5];
    jacobi_eig(A, V, 3, 8);
    double m0 = fabs(A[0]), m1 = fabs(A[4]), m2 = fabs(A[8]);
    int z = 0;
    if (m1 < m0) z = 1;
    if (m2 < (z == 0 ? m0 : m1)) z = 2;
    int e0 = z == 0 ? 1 : 0, e1 = z == 2 ? 1 : 2;
    double me0 = e0 == 0 ? m0 : m1, me1 = e1 == 1 ? m1 : m2;
    if (me1 > me0) { int tmp = e0; e0 = e1; e1 = tmp; }
    double L0 = A[4 * e0], L1 = A[4 * e1];
    double v = sqrt(fmax(0.0, -L1 / L0));
    double Ls[4][3];
    int n = 0;
    p3p_line(v, V, e0, e1, a12, a13, a23, b12, b13, b23, Ls, &n);
    p3p_line(-v, V, e0, e1, a12, a13, a23, b12, b13, b23, Ls, &n);
    double cx0 = d12[1] * d13[2] - d12[2] * d13[1];
    double cx1 = d12[2] * d13[0] - d12[0] * d13[2];
    double cx2 = d12[0] * d13[1] - d12[1] * d13[0];
    double m[9] = {d12[0], d13[0], cx0, d12[1], d13[1], cx1, d12[2], d13[2], cx2}, mi[9];
    {
        double c00 = m[4] * m[8] - m[5] * m[7], c01 = m[5] * m[6] - m[3] * m[8], c02 = m[3] * m[7] - m[4] * m[6];
        double id = 1.0 / (m[0] * c00 + m[1] * c01 + m[2] * c02);
        mi[0] = c00 * id; mi[1] = (m[2] * m[7] - m[1] * m[8]) * id; mi[2] = (m[1] * m[5] - m[2] * m[4]) * id;
        mi[3] = c01 * id; mi[4] = (m[0] * m[8] - m[2] * m[6]) * id; mi[5] = (m[2] * m[3] - m[0] * m[5]) * id;
        mi[6] = c02 * id; mi[7] = (m[1] * m[6] - m[0] * m[7]) * id; mi[8] = (m[0] * m[4] - m[1] * m[3]) * id;
    }
    int kept = 0;
    for (int r = 0; r < n && r < 4; ++r) {
        double L[3] = {Ls[r][0], Ls[r][1], Ls[r][2]};
        p3p_refine_depths(L, a12, a13, a23, b12, b13, b23);
        if (!(L[0] > 0.0) || !(L[1] > 0.0) || !(L[2] > 0.0) || !pnp_finite(L[0]) || !pnp_finite(L[1]) || !pnp_finite(L[2])) continue;
        double ry[3][3], yd1[3], yd2[3], P[12];
        for (int k = 0; k < 3; ++k)
            for (int c = 0; c < 3; ++c) ry[k][c] = y[k][c] * L[k];
        for (int c = 0; c < 3; ++c) {
            yd1[c] = ry[0][c] - ry[1][c];
            yd2[c] = ry[0][c] - ry[2][c];
        }
        double yx0 = yd1[1] * yd2[2] - yd1[2] * yd2[1];
        double yx1 = yd1[2] * yd2[0] - yd1[0] * yd2[2];
        double yx2 = yd1[0] * yd2[1] - yd1[1] * yd2[0];
        double Y[9] = {yd1[0], yd2[0], yx0, yd1[1], yd2[1], yx1, yd1[2], yd2[2], yx2};
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) P[3 * i + j] = Y[3 * i] * mi[j] + Y[3 * i + 1] * mi[3 + j] + Y[3 * i + 2] * mi[6 + j];
        for (int i = 0; i < 3; ++i) P[9 + i] = ry[0][i] - (P[3 * i] * X[0] + P[3 * i + 1] * X[1] + P[3 * i + 2] * X[2]);
        int ok = 1;
        for (int i = 0; i < 12; ++i) ok = ok && pnp_finite(P[i]);
        if (!ok) continue;
        memcpy(out + 12 * kept, P, sizeof P);
        ++kept;
    }
    return kept;
}

/* ---------------------------------------------------------------- refinement (kernel twins: add_gn, gn_step) */
static void to_camera(const double* P, double fx, double fy, pnp_camera* K)
{
    K->fx = fx; K->fy = fy;
    for (int i = 0; i < 9; ++i) K->r[i] = P[i];
    for (int i = 0; i < 3; ++i) K->t[i] = P[9 + i];
}

static void add_gn(double* v, const pnp_camera* K, double x, double y, const double* Xw)
{
    double q0 = K->r[0] * Xw[0] + K->r[1] * Xw[1] + K->r[2] * Xw[2];
    double q1 = K->r[3] * Xw[0] + K->r[4] * Xw[1] + K->r[5] * Xw[2];
    double q2 = K->r[6] * Xw[0] + K->r[7] * Xw[1] + K->r[8] * Xw[2];
    double p0 = q0 + K->t[0], p1 = q1 + K->t[1], p2 = q2 + K->t[2];
    double iz = 1.0 / p2;
    double u0 = p0 * iz, u1 = p1 * iz;
    double ex = (u0 - x) * K->fx, ey = (u1 - y) * K->fy;
    double a0 = K->fx * iz, a2 = -(a0 * u0);
    double b1 = K->fy * iz, b2 = -(b1 * u1);
    double ju[6] = {a2 * p1, a0 * p2 - a2 * p0, -(a0 * p1), a0, 0.0, a2};
    double jv[6] = {b2 * p1 - b1 * p2, -(b2 * p0), b1 * p0, 0.0, b1, b2};
    int e = 0;
    for (int i = 0; i < 6; ++i)
        for (int j = i; j < 6; ++j) {
            v[e] = v[e] + ju[i] * ju[j];
            v[e] = v[e] + jv[i] * jv[j];
            ++e;
        }
    for (int i = 0; i < 6; ++i) {
        v[21 + i] = v[21 + i] + ju[i] * ex;
        v[21 + i] = v[21 + i] + jv[i] * ey;
    }
    v[27] = v[27] + (ex * ex + ey * ey);
}

static int gn_step(const double* v, const pnp_camera* K, pnp_camera* O)
{
    double H[36], L[36], inv[6], z[6], dl[6];
    int e = 0;
    for (int i = 0; i < 6; ++i)
        for (int j = i; j < 6; ++j) {
            H[i * 6 + j] = v[e];
            H[j * 6 + i] = v[e];
            ++e;
        }
    for (int j = 0; j < 6; ++j) {
        double s = H[j * 6 + j];
        for (int k = 0; k < j; ++k) s = s - L[j * 6 + k] * L[j * 6 + k];
        if (!(s > 0.0)) return 0;
        double d = sqrt(s);
        inv[j] = 1.0 / d;
        for (int i = j + 1; i < 6; ++i) {
            double w = H[i * 6 + j];
            for (int k = 0; k < j; ++k) w = w - L[i * 6 + k] * L[j * 6 + k];
            L[i * 6 + j] = w * inv[j];
        }
        L[j * 6 + j] = d;
    }
    for (int i = 0; i < 6; ++i) {
        double w = -v[21 + i];
        for (int k = 0; k < i; ++k) w = w - L[i * 6 + k] * z[k];
        z[i] = w * inv[i];
    }
    for (int i = 5; i >= 0; --i) {
        double w = z[i];
        for (int k = i + 1; k < 6; ++k) w = w - L[k * 6 + i] * dl[k];
        dl[i] = w * inv[i];
    }
    double hx = 0.5 * dl[0], hy = 0.5 * dl[1], hz = 0.5 * dl[2];
    double in = 1.0 / sqrt(1.0 + hx * hx + hy * hy + hz * hz);
    double qw = in, qx = hx * in, qy = hy * in, qz = hz * in;
    double D[9] = {1.0 - 2.0 * (qy * qy + qz * qz), 2.0 * (qx * qy - qw * qz), 2.0 * (qx * qz + qw * qy),
                   2.0 * (qx * qy + qw * qz), 1.0 - 2.0 * (qx * qx + qz * qz), 2.0 * (qy * qz - qw * qx),
                   2.0 * (qx * qz - qw * qy), 2.0 * (qy * qz + qw * qx), 1.0 - 2.0 * (qx * qx + qy * qy)};
    O->fx = K->fx; O->fy = K->fy;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) O->r[3 * i + j] = D[3 * i] * K->r[j] + D[3 * i + 1] * K->r[3 + j] + D[3 * i + 2] * K->r[6 + j];
    for (int i = 0; i < 3; ++i) O->t[i] = (D[3 * i] * K->t[0] + D[3 * i + 1] * K->t[1] + D[3 * i + 2] * K->t[2]) + dl[3 + i];
    return 1;
}

typedef struct {
    const double* nx;        /* [M] normalised coordinates */
    const double* ny;
    const double* X;         /* [M, 3] */
    int M;
    double thr2;
} pnp_query;

static int pnp_count(const pnp_query* Q, const pnp_camera* K, uint8_t* mask)
{
    int n = 0;
    for (int i = 0; i < Q->M; ++i) {
        double e2;
        int in = pnp_reproject(K, Q->X + 3 * (size_t)i, Q->nx[i], Q->ny[i], Q->thr2, &e2);
        if (mask) mask[i] = (uint8_t)in;
        n += in;
    }
    return n;
}

/* The block sums of the kernel: lane t sums correspondences t, t + 256, ... in order, lane_tree adds the lanes. */
static void pnp_gn_sums(const pnp_query* Q, const uint8_t* mask, const pnp_camera* K, double* part /* [PNP_SUMS][256] */,
                        double* v)
{
    for (int t = 0; t < SFM_RANSAC_LANES; ++t) {
        double s[PNP_SUMS];
        for (int e = 0; e < PNP_SUMS; ++e) s[e] = 0.0;
        for (int i = t; i < Q->M; i += SFM_RANSAC_LANES)
            if (mask[i]) add_gn(s, K, Q->nx[i], Q->ny[i], Q->X + 3 * (size_t)i);
        for (int e = 0; e < PNP_SUMS; ++e) part[e * SFM_RANSAC_LANES + t] = s[e];
    }
    for (int e = 0; e < PNP_SUMS; ++e) v[e] = lane_tree(part + e * SFM_RANSAC_LANES);
}

static double pnp_cost(const pnp_query* Q, const uint8_t* mask, const pnp_camera* K, double* part)
{
    for (int t = 0; t < SFM_RANSAC_LANES; ++t) {
        double s = 0.0;
        for (int i = t; i < Q->M; i += SFM_RANSAC_LANES)
            if (mask[i]) {
                double e2;
                pnp_reproject(K, Q->X + 3 * (size_t)i, Q->nx[i], Q->ny[i], Q->thr2, &e2);
                s = s + e2;
            }
        part[t] = s;
    }
    return lane_tree(part);
}

/* Arguments as sfm_pnp_ransac (out_iters may be NULL).  Returns 0, or -1 when the scratch allocation fails. */
int sfm_oracle_pnp_ransac(int n_images, const double* cams, const int32_t* image, int n_query, const float* xy, const double* X,
                          int stride, const int32_t* count, const sfm_pnp_params* prm, double* out_pose, int32_t* out_ninl,
                          uint8_t* out_status, uint8_t* out_mask, int32_t* out_iters, int64_t* out_counts)
{
    const double thr2 = prm->max_error * prm->max_error;
    double* nx = (double*)malloc(sizeof(double) * (size_t)stride);
    double* ny = (double*)malloc(sizeof(double) * (size_t)stride);
    double* part = (double*)malloc(sizeof(double) * PNP_SUMS * SFM_RANSAC_LANES);
    if (!nx || !ny || !part) {
        free(nx); free(ny); free(part);
        return -1;
    }
    for (int s = 0; s < 5; ++s) out_counts[s] = 0;
    for (int q = 0; q < n_query; ++q) {
        const int64_t base = (int64_t)q * stride;
        uint8_t* mask = out_mask + base;
        const int img = image[q];
        double fx = 0.0, fy = 0.0, cx = 0.0, cy = 0.0;
        int status = 0, M = 0, cur = 0, done = 0;
        double best[12];
        if (img < 0 || img >= n_images) {
            status = 4;
        } else {
            const double* c = cams + 16 * (size_t)img;
            fx = c[0]; fy = c[1]; cx = c[2]; cy = c[3];
            if (!(fx > 0.0) || !(fy > 0.0) || !pnp_finite(fx) || !pnp_finite(fy)) status = 4;
        }
        if (status == 0) {
            M = count[q] < 0 ? 0 : (count[q] > stride ? stride : count[q]);
            if (M < 3) status = 1;
        }
        const pnp_query Q = {nx, ny, X + 3 * base, M, thr2};
        memset(mask, 0, (size_t)stride);
        if (status == 0) {
            for (int i = 0; i < M; ++i) {
                nx[i] = ((double)xy[2 * (base + i)] - cx) / fx;
                ny[i] = ((double)xy[2 * (base + i) + 1] - cy) / fy;
            }
            int best_n = -1;
            while (done < prm->max_iters) {
                int nb = ransac_batch(done);
                if (nb > prm->max_iters - done) nb = prm->max_iters - done;
                for (int h = 0; h < nb; ++h) {
                    int idx[3];
                    draw_sample(prm->seed, (uint32_t)img, (uint32_t)(done + h), 3, M, idx);
                    double sx[3], sy[3], sX[9], poses[48];
                    for (int k = 0; k < 3; ++k) {
                        sx[k] = nx[idx[k]]; sy[k] = ny[idx[k]];
                        for (int c = 0; c < 3; ++c) sX[3 * k + c] = Q.X[3 * (size_t)idx[k] + c];
                    }
                    int nr = sfm_oracle_p3p(sx, sy, sX, poses);
                    for (int r = 0; r < nr; ++r) {
                        pnp_camera K;
                        to_camera(poses + 12 * r, fx, fy, &K);
                        int n = pnp_count(&Q, &K, NULL);
                        if (n > best_n) { best_n = n; memcpy(best, poses + 12 * r, sizeof best); }
                    }
                }
                done += nb;
                if (should_stop(best_n, M, 3, done, prm->confidence)) break;
            }
            cur = best_n;
            if (cur < 0) {
                status = 2;
            } else {
                pnp_camera P;
                to_camera(best, fx, fy, &P);
                for (int round = 0; round < SFM_LO_ROUNDS && prm->refine_iters > 0 && cur >= 3; ++round) {
                    pnp_count(&Q, &P, mask);
                    pnp_camera it = P;
                    int moved = 0;
                    for (int s = 0; s < prm->refine_iters; ++s) {
                        double v[PNP_SUMS];
                        pnp_gn_sums(&Q, mask, &it, part, v);
                        pnp_camera nxt;
                        if (!gn_step(v, &it, &nxt)) break;
                        if (!(pnp_cost(&Q, mask, &nxt, part) < v[27])) break;
                        it = nxt;
                        moved = 1;
                    }
                    if (!moved) break;
                    int n = pnp_count(&Q, &it, NULL);
                    if (n < cur) break;
                    cur = n;
                    P = it;
                }
                if (cur < prm->min_inliers || (double)cur < prm->min_inlier_ratio * (double)M) status = 3;
                for (int i = 0; i < 9; ++i) best[i] = P.r[i];
                for (int i = 0; i < 3; ++i) best[9 + i] = P.t[i];
            }
        }
        if (status == 0) {
            pnp_camera P;
            to_camera(best, fx, fy, &P);
            pnp_count(&Q, &P, mask);
            for (int i = M; i < stride; ++i) mask[i] = 0;
        } else {
            memset(mask, 0, (size_t)stride);
        }
        for (int i = 0; i < 12; ++i) out_pose[12 * (size_t)q + i] = status == 0 ? best[i] : 0.0;
        out_ninl[q] = (status == 0 || status == 3) ? cur : 0;
        out_status[q] = (uint8_t)status;
        if (out_iters) out_iters[q] = done;
        out_counts[status] += 1;
    }
    free(nx); free(ny); free(part);
    return 0;
}
