// eval_metrics.h -- per-frame imitation metrics of one recorded trajectory row, fp64, host/device portable (the CUDA metric kernel in
// eval.cu and the CPU test in tests/test_eval_metrics_cpu.py compile the same code).  Restates uhc_b200/metrics.py, which restates the
// reference's smpl_eval.compute_metrics (uhc/smpllib/smpl_eval.py:24-123): millimetres, 24 SMPL joints, Pelvis = joint 0.
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define UHC_HD __host__ __device__ inline
#else
#define UHC_HD inline
#endif

namespace uhc_eval {

constexpr int NJ = 24;
// columns of a frame_metrics row (include/uhc_eval.h)
constexpr int M_ROOT = 0, M_MPJPE = 1, M_MPJPE_G = 2, M_PA_MPJPE = 3, M_VEL = 4, M_ACCEL = 5, NMET = 6;

// transformation.py quaternion_matrix: (w, x, y, z), normalised by |q|^2; identity below 4 eps
UHC_HD void quat_mat3(const double q[4], double R[9]) {
    const double n = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
    if (!(n > 4.0 * 2.220446049250313e-16)) { for (int i = 0; i < 9; i++) R[i] = (i % 4) == 0 ? 1.0 : 0.0; return; }
    const double s = 2.0 / n, w = q[0], x = q[1], y = q[2], z = q[3];
    R[0] = 1 - s * (y * y + z * z); R[1] = s * (x * y - z * w); R[2] = s * (x * z + y * w);
    R[3] = s * (x * y + z * w); R[4] = 1 - s * (x * x + z * z); R[5] = s * (y * z - x * w);
    R[6] = s * (x * z - y * w); R[7] = s * (y * z + x * w); R[8] = 1 - s * (x * x + y * y);
}

// ||I - X_pred X_gt^-1||_F with X = [R t; 0 1] (X_gt^-1 = [R^T, -R^T t]), in metres (not yet divided by the frame count)
template <class P, class G>
UHC_HD double root_frob(const P *qp, const G *qg) {
    double a[4], b[4], Rp[9], Rg[9];
    for (int i = 0; i < 4; i++) { a[i] = (double)qp[3 + i]; b[i] = (double)qg[3 + i]; }
    quat_mat3(a, Rp); quat_mat3(b, Rg);
    double acc = 0.0, RR[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            double s = 0.0;
            for (int k = 0; k < 3; k++) s += Rp[3 * i + k] * Rg[3 * j + k];      // Rp Rg^T
            RR[3 * i + j] = s;
            const double e = (i == j ? 1.0 : 0.0) - s;
            acc += e * e;
        }
    for (int i = 0; i < 3; i++) {          // translation column: t_p - Rp Rg^T t_g
        double s = 0.0;
        for (int k = 0; k < 3; k++) s += RR[3 * i + k] * (double)qg[k];
        const double e = (double)qp[i] - s;
        acc += e * e;
    }
    return sqrt(acc);
}

// 3x3 SVD A = U diag(s) V^T (row-major), one-sided Jacobi on the columns of A; s sorted descending as numpy.linalg.svd returns it
UHC_HD void svd3(const double A[9], double U[9], double s[3], double V[9]) {
    double B[9];
    for (int i = 0; i < 9; i++) { B[i] = A[i]; V[i] = (i % 4) == 0 ? 1.0 : 0.0; }
    for (int sweep = 0; sweep < 30; sweep++) {
        double off = 0.0;
        for (int pq = 0; pq < 3; pq++) {
            const int p = pq == 2 ? 1 : 0, q = pq == 0 ? 1 : 2;
            double al = 0.0, be = 0.0, ga = 0.0;
            for (int i = 0; i < 3; i++) { al += B[3 * i + p] * B[3 * i + p]; be += B[3 * i + q] * B[3 * i + q]; ga += B[3 * i + p] * B[3 * i + q]; }
            if (ga == 0.0 || fabs(ga) <= 1e-17 * sqrt(al * be)) continue;
            off = fmax(off, fabs(ga) / sqrt(al * be));
            const double zeta = (be - al) / (2.0 * ga);
            const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
            const double c = 1.0 / sqrt(1.0 + t * t), sn = c * t;
            for (int i = 0; i < 3; i++) {
                const double bp = B[3 * i + p], bq = B[3 * i + q];
                B[3 * i + p] = c * bp - sn * bq; B[3 * i + q] = sn * bp + c * bq;
                const double vp = V[3 * i + p], vq = V[3 * i + q];
                V[3 * i + p] = c * vp - sn * vq; V[3 * i + q] = sn * vp + c * vq;
            }
        }
        if (off <= 1e-16) break;
    }
    int ord[3] = {0, 1, 2};
    double nrm[3];
    for (int j = 0; j < 3; j++) nrm[j] = sqrt(B[j] * B[j] + B[3 + j] * B[3 + j] + B[6 + j] * B[6 + j]);
    for (int a = 0; a < 2; a++)
        for (int b = a + 1; b < 3; b++)
            if (nrm[ord[b]] > nrm[ord[a]]) { const int tmp = ord[a]; ord[a] = ord[b]; ord[b] = tmp; }
    double Vs[9];
    for (int j = 0; j < 3; j++) {
        const int c = ord[j];
        s[j] = nrm[c];
        for (int i = 0; i < 3; i++) { Vs[3 * i + j] = V[3 * i + c]; U[3 * i + j] = s[j] > 0.0 ? B[3 * i + c] / s[j] : 0.0; }
    }
    for (int i = 0; i < 9; i++) V[i] = Vs[i];
    // rank-deficient input: complete U to an orthonormal basis (the singular value is 0, so only the basis matters)
    const double tiny = 1e-300 + 1e-15 * s[0];
    if (!(s[1] > tiny)) {   // any unit vector orthogonal to U0
        const double ax = fabs(U[0]), ay = fabs(U[3]), az = fabs(U[6]);
        double e[3] = {0, 0, 0}; e[ax <= ay && ax <= az ? 0 : (ay <= az ? 1 : 2)] = 1.0;
        if (!(s[0] > tiny)) { U[0] = 1; U[3] = 0; U[6] = 0; e[0] = 0; e[1] = 1; e[2] = 0; }
        double u1[3] = {U[3] * e[2] - U[6] * e[1], U[6] * e[0] - U[0] * e[2], U[0] * e[1] - U[3] * e[0]};
        const double n = sqrt(u1[0] * u1[0] + u1[1] * u1[1] + u1[2] * u1[2]);
        for (int i = 0; i < 3; i++) U[3 * i + 1] = u1[i] / n;
    }
    if (!(s[2] > tiny)) {   // U2 = U0 x U1
        U[2] = U[3] * U[7] - U[6] * U[4]; U[5] = U[6] * U[1] - U[0] * U[7]; U[8] = U[0] * U[4] - U[3] * U[1];
    }
}

UHC_HD double det3(const double M[9]) {
    return M[0] * (M[4] * M[8] - M[5] * M[7]) - M[1] * (M[3] * M[8] - M[5] * M[6]) + M[2] * (M[3] * M[7] - M[4] * M[6]);
}

// metrics.py procrustes_mpjpe for one frame: mean joint error after the best similarity alignment of pred onto gt, both [NJ][3]
UHC_HD double pa_mpjpe(const double (*pr)[3], const double (*gt)[3]) {
    double mp[3] = {0, 0, 0}, mg[3] = {0, 0, 0};
    for (int j = 0; j < NJ; j++) for (int k = 0; k < 3; k++) { mp[k] += pr[j][k]; mg[k] += gt[j][k]; }
    for (int k = 0; k < 3; k++) { mp[k] /= NJ; mg[k] /= NJ; }
    double np2 = 0.0, ng2 = 0.0;
    for (int j = 0; j < NJ; j++) for (int k = 0; k < 3; k++) { const double a = pr[j][k] - mp[k], b = gt[j][k] - mg[k]; np2 += a * a; ng2 += b * b; }
    const double npd = sqrt(np2), ng = sqrt(ng2);
    double K[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};      // K = G^T P of the centred, normalised sets
    for (int j = 0; j < NJ; j++)
        for (int a = 0; a < 3; a++)
            for (int b = 0; b < 3; b++) K[3 * a + b] += ((gt[j][a] - mg[a]) / ng) * ((pr[j][b] - mp[b]) / npd);
    double U[9], s[3], V[9];
    svd3(K, U, s, V);
    // no reflections: flip the last column of V (and the last singular value) when det(V U^T) < 0
    const double d = det3(V) * det3(U) < 0.0 ? -1.0 : 1.0;
    for (int i = 0; i < 3; i++) V[3 * i + 2] *= d;
    s[2] *= d;
    double R[9];           // R = V U^T
    for (int a = 0; a < 3; a++)
        for (int b = 0; b < 3; b++) R[3 * a + b] = V[3 * a] * U[3 * b] + V[3 * a + 1] * U[3 * b + 1] + V[3 * a + 2] * U[3 * b + 2];
    const double scale = (s[0] + s[1] + s[2]) * ng / npd;
    double mpR[3];
    for (int b = 0; b < 3; b++) mpR[b] = mp[0] * R[b] + mp[1] * R[3 + b] + mp[2] * R[6 + b];
    double err = 0.0;
    for (int j = 0; j < NJ; j++) {
        double e2 = 0.0;
        for (int b = 0; b < 3; b++) {
            const double pR = pr[j][0] * R[b] + pr[j][1] * R[3 + b] + pr[j][2] * R[6 + b];
            const double al = scale * pR + (mg[b] - scale * mpR[b]);
            e2 += (al - gt[j][b]) * (al - gt[j][b]);
        }
        err += sqrt(e2);
    }
    return err / NJ;
}

// mean over joints of ||(a0 - a1 [+ a2 ...]) - (b0 - ...)||: the finite-difference errors (vel: rows t-1, t; accel: t-2, t-1, t)
template <class P, class G>
UHC_HD double fd_err(const P *p0, const P *p1, const P *p2, const G *g0, const G *g1, const G *g2) {
    double acc = 0.0;
    for (int j = 0; j < NJ; j++) {
        double e2 = 0.0;
        for (int k = 0; k < 3; k++) {
            const int i = 3 * j + k;
            const double dp = p2 ? (double)p2[i] - 2.0 * (double)p1[i] + (double)p0[i] : (double)p0[i] - (double)p1[i];
            const double dg = g2 ? (double)g2[i] - 2.0 * (double)g1[i] + (double)g0[i] : (double)g0[i] - (double)g1[i];
            e2 += (dp - dg) * (dp - dg);
        }
        acc += sqrt(e2);
    }
    return acc / NJ;
}

// the six metrics of row t of a clip with `nframes` recorded rows.  qp / qg: qpos rows (root position + quaternion read);
// jp[0..2] / jg[0..2]: world joint positions [72] of rows t, t-1, t-2 (null where the row does not exist).  vel is defined from the
// clip's 2nd row on, accel from its 3rd; the others are NaN-free for every row.  out in mm.
template <class P, class G>
UHC_HD void frame_metrics(const P *qp, const G *qg, const P *const jp[3], const G *const jg[3], int nframes, double out[NMET]) {
    const double nan = NAN;
    out[M_ROOT] = root_frob(qp, qg) / (double)nframes * 1000.0;
    double pr[NJ][3], gt[NJ][3], eg = 0.0, el = 0.0;
    for (int j = 0; j < NJ; j++) {
        double d2 = 0.0, l2 = 0.0;
        for (int k = 0; k < 3; k++) {
            const double a = (double)jp[0][3 * j + k], b = (double)jg[0][3 * j + k];
            d2 += (a - b) * (a - b);
            pr[j][k] = a - (double)jp[0][k]; gt[j][k] = b - (double)jg[0][k];      // Pelvis-relative
            l2 += (pr[j][k] - gt[j][k]) * (pr[j][k] - gt[j][k]);
        }
        eg += sqrt(d2); el += sqrt(l2);
    }
    out[M_MPJPE_G] = eg / NJ * 1000.0;
    out[M_MPJPE] = el / NJ * 1000.0;
    out[M_PA_MPJPE] = pa_mpjpe(pr, gt) * 1000.0;
    out[M_VEL] = jp[1] ? fd_err<P, G>(jp[0], jp[1], nullptr, jg[0], jg[1], nullptr) * 1000.0 : nan;
    out[M_ACCEL] = jp[2] ? fd_err<P, G>(jp[0], jp[1], jp[2], jg[0], jg[1], jg[2]) * 1000.0 : nan;
}

}  // namespace uhc_eval
