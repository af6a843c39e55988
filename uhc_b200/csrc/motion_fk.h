// motion_fk.h -- one frame of the expert table from raw SMPL input, fp64, host/device portable (the CUDA kernel of motion_lib.cu and the
// CPU test in tests/test_motion_fk_cpu.py compile the same code).  Restates uhc_b200/motion_lib.py make_expert = qpos_fk(smpl_to_qpos(...)):
//   smpl_to_qpos  scipy Rotation.from_rotvec + as_euler("ZYX") per SMPL joint, SMPL -> depth-first body order, root quaternion (w >= 0),
//                 root position = trans + the model's root offset
//   qpos_fk       local quaternions (euler_zyx_quat), tree FK, finite-difference qvel / body angular velocity at 30 Hz
// Every operation keeps the order of the numpy code, so a build without FMA contraction differs from it only where the libm and CUDA
// transcendentals differ (a few ulp).  Frame t >= 1 differences against frame t - 1, frame 0 against frame 1 (qvel[:1] repeated); both
// frames are recomputed from their input rows, so frames are independent of each other.
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define UHC_MHD __host__ __device__ inline
#else
#define UHC_MHD inline
#endif

namespace uhc_motion {

constexpr int NB = 24, NQ = 76, NV = 75, REC = 576;
// record layout (include/uhc_b200.h UHC_EX_SIZE): qpos76 qvel75 wbpos72 wbquat96 bquat96 bangvel72 ee_wpos15 body_com72 pad2
constexpr int R_QPOS = 0, R_QVEL = 76, R_WBPOS = 151, R_WBQUAT = 223, R_BQUAT = 319, R_BANGVEL = 415, R_EE = 487, R_BCOM = 502, R_PAD = 574;
constexpr double PI = 3.141592653589793;
constexpr double DT = 1.0 / 30;
// trans of a clip without one (smpl_to_qpos: trans = None)
constexpr double DEFAULT_TRANS_Z = 0.91437225;
// SMPL joint of every model body: SMPL_BONE_ORDER_NAMES.index(body_names[b]) for the depth-first SMPL humanoid
UHC_MHD int smpl_joint(int b) {
    const int j[NB] = {0, 1, 4, 7, 10, 2, 5, 8, 11, 3, 6, 9, 12, 15, 13, 16, 18, 20, 22, 14, 17, 19, 21, 23};
    return j[b];
}

// kinematic tables of one body-shape variant
struct Kin {
    const double *off_ipos;   // [24][6]: body offset in the parent frame (body 0: the root offset), centre of mass in the body frame
    const int *parent;        // [24], parent[0] = -1
    const int *ee;            // [5] end-effector bodies
};

// quaternions are (w, x, y, z) as in motion_lib.py; scipy's are (x, y, z, w)
UHC_MHD void qmul(const double *a, const double *b, double *o) {
    const double w0 = a[0], x0 = a[1], y0 = a[2], z0 = a[3], w1 = b[0], x1 = b[1], y1 = b[2], z1 = b[3];
    o[0] = w0 * w1 - x0 * x1 - y0 * y1 - z0 * z1;
    o[1] = w0 * x1 + x0 * w1 + y0 * z1 - z0 * y1;
    o[2] = w0 * y1 - x0 * z1 + y0 * w1 + z0 * x1;
    o[3] = w0 * z1 + x0 * y1 - y0 * x1 + z0 * w1;
}
UHC_MHD void qinv(const double *q, double *o) {
    const double n = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
    o[0] = q[0] / n; o[1] = -q[1] / n; o[2] = -q[2] / n; o[3] = -q[3] / n;
}
UHC_MHD void cross(const double *a, const double *b, double *o) {
    o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0];
}
// v + 2 (w (u x v) + u x (u x v))
UHC_MHD void qrot(const double *q, const double *v, double *o) {
    double uv[3], uuv[3];
    cross(q + 1, v, uv); cross(q + 1, uv, uuv);
    for (int i = 0; i < 3; i++) o[i] = v[i] + 2 * (q[0] * uv[i] + uuv[i]);
}
// quaternion_from_euler(e0, e1, e2, 'rzyx') = Rz(e0) Ry(e1) Rx(e2)
UHC_MHD void euler_zyx_quat(const double *e, double *o) {
    const double h0 = 0.5 * e[0], h1 = 0.5 * e[1], h2 = 0.5 * e[2];
    const double qz[4] = {cos(h0), 0.0, 0.0, sin(h0)}, qy[4] = {cos(h1), 0.0, sin(h1), 0.0}, qx[4] = {cos(h2), sin(h2), 0.0, 0.0};
    double t[4];
    qmul(qz, qy, t); qmul(t, qx, o);
}
// rotation_from_quaternion_batch: axis * angle, the arccos argument clamped to 1 - 1e-7, identity below |sin| 1e-5
UHC_MHD void rot_from_quat(const double *q, double axis[3], double *angle) {
    double w = q[0];
    w = w < -1.0 + 1e-7 ? -1.0 + 1e-7 : (w > 1.0 - 1e-7 ? 1.0 - 1e-7 : w);
    const double ac = acos(w), sn = sin(ac);
    if (fabs(sn) < 1e-5) { axis[0] = 1.0; axis[1] = 0.0; axis[2] = 0.0; *angle = 0.0; return; }
    for (int i = 0; i < 3; i++) axis[i] = q[1 + i] / sn;
    *angle = 2 * ac;
}

// scipy Rotation.from_rotvec(v).as_quat(): (x, y, z, w), Taylor series of sin(a/2)/a at angles <= 1e-3
UHC_MHD void rotvec_quat_xyzw(const double *v, double *q) {
    const double a = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
    double s;
    if (a <= 1e-3) { const double a2 = a * a; s = 0.5 - a2 / 48 + a2 * a2 / 3840; }
    else s = sin(a / 2) / a;
    q[0] = s * v[0]; q[1] = s * v[1]; q[2] = s * v[2]; q[3] = cos(a / 2);
}
// scipy Rotation.as_euler("ZYX") (intrinsic) on an (x, y, z, w) quaternion: the quaternion method of Bernardes & Viollet for the reversed
// extrinsic sequence "xyz" (axes i, j, k = 0, 1, 2, even permutation); at gimbal lock (middle angle within 1e-7 of 0 or pi before the
// Tait-Bryan shift) the last intrinsic angle is set to zero.  Angles wrapped into [-pi, pi].
UHC_MHD void quat_euler_zyx(const double *q, double *e) {
    const double x = q[0], y = q[1], z = q[2], w = q[3];
    const double a = w - y, b = x + z, c = y + w, d = z - x;
    double ang[3];
    ang[1] = 2 * atan2(hypot(c, d), hypot(a, b));
    int degenerate = 0;
    if (fabs(ang[1]) <= 1e-7) degenerate = 1;
    else if (fabs(ang[1] - PI) <= 1e-7) degenerate = 2;
    const double half_sum = atan2(b, a), half_diff = atan2(d, c);
    if (degenerate == 0) { ang[0] = half_sum - half_diff; ang[2] = half_sum + half_diff; }
    else { ang[0] = 0.0; ang[2] = degenerate == 1 ? 2 * half_sum : 2 * half_diff; }
    ang[1] -= PI / 2;
    e[0] = ang[2]; e[1] = ang[1]; e[2] = ang[0];
    for (int i = 0; i < 3; i++) {
        if (e[i] < -PI) e[i] += 2 * PI;
        else if (e[i] > PI) e[i] -= 2 * PI;
    }
}

// smpl_to_qpos for one row: pose = pose_dim (72, or 156 = SMPL-H: columns 66.. are the hands, replaced by zero), trans = 3 values or
// null (DEFAULT_TRANS_Z above the origin); root_off = the variant's root offset
UHC_MHD void frame_qpos(const double *pose, int pose_dim, const double *trans, const double *root_off, double *qpos) {
    const int keep = pose_dim == 156 ? 66 : 72;
    const double tr[3] = {trans ? trans[0] : 0.0, trans ? trans[1] : 0.0, trans ? trans[2] : DEFAULT_TRANS_Z};
    for (int i = 0; i < 3; i++) qpos[i] = tr[i] + root_off[i];
    for (int b = 0; b < NB; b++) {
        const int j = smpl_joint(b);
        const double v[3] = {3 * j < keep ? pose[3 * j] : 0.0, 3 * j < keep ? pose[3 * j + 1] : 0.0, 3 * j < keep ? pose[3 * j + 2] : 0.0};
        double q[4];
        rotvec_quat_xyzw(v, q);
        if (b == 0) {
            const double sg = q[3] < 0 ? -1.0 : 1.0;
            qpos[3] = sg * q[3]; qpos[4] = sg * q[0]; qpos[5] = sg * q[1]; qpos[6] = sg * q[2];
        } else {
            quat_euler_zyx(q, qpos + 7 + 3 * (b - 1));
        }
    }
}
// bquat: the root quaternion, then the local quaternion of every joint
UHC_MHD void frame_bquat(const double *qpos, double *bq) {
    for (int i = 0; i < 4; i++) bq[i] = qpos[3 + i];
    for (int b = 1; b < NB; b++) euler_zyx_quat(qpos + 7 + 3 * (b - 1), bq + 4 * b);
}

// the record of frame t of a clip of at least 2 rows: pose / trans point at the clip's row 0 (trans may be null); Out = float or double
template <class Out>
UHC_MHD void expert_frame(const double *pose, int pose_dim, const double *trans, int t, const Kin &k, Out *rec) {
    const int f0 = t == 0 ? 0 : t - 1, f1 = t == 0 ? 1 : t;    // (cur, nxt) of the finite differences
    double qc[NQ], qn[NQ], bc[4 * NB], bn[4 * NB];
    frame_qpos(pose + (size_t)f0 * pose_dim, pose_dim, trans ? trans + 3 * (size_t)f0 : nullptr, k.off_ipos, qc);
    frame_qpos(pose + (size_t)f1 * pose_dim, pose_dim, trans ? trans + 3 * (size_t)f1 : nullptr, k.off_ipos, qn);
    frame_bquat(qc, bc); frame_bquat(qn, bn);
    const double *q = t == 0 ? qc : qn, *bq = t == 0 ? bc : bn;
    // tree FK (bodies are numbered depth-first: a parent precedes its children)
    double wpos[3 * NB], wquat[4 * NB];
    for (int b = 0; b < NB; b++) {
        if (b == 0) { for (int i = 0; i < 3; i++) wpos[i] = q[i]; for (int i = 0; i < 4; i++) wquat[i] = q[3 + i]; }
        else {
            const int p = k.parent[b];
            double r[3];
            qrot(wquat + 4 * p, k.off_ipos + 6 * b, r);
            for (int i = 0; i < 3; i++) wpos[3 * b + i] = r[i] + wpos[3 * p + i];
            qmul(wquat + 4 * p, bq + 4 * b, wquat + 4 * b);
        }
        double c[3];
        qrot(wquat + 4 * b, k.off_ipos + 6 * b + 3, c);
        for (int i = 0; i < 3; i++) rec[R_BCOM + 3 * b + i] = (Out)(c[i] + wpos[3 * b + i]);
    }
    for (int i = 0; i < NQ; i++) rec[R_QPOS + i] = (Out)q[i];
    for (int i = 0; i < 3 * NB; i++) rec[R_WBPOS + i] = (Out)wpos[i];
    for (int i = 0; i < 4 * NB; i++) { rec[R_WBQUAT + i] = (Out)wquat[i]; rec[R_BQUAT + i] = (Out)bq[i]; }
    for (int e = 0; e < 5; e++) for (int i = 0; i < 3; i++) rec[R_EE + 3 * e + i] = (Out)wpos[3 * k.ee[e] + i];
    // get_qvel_fd_batch: linear velocity, root angular velocity in the body frame (angle wrapped into [-pi, pi]), joint angle rates
    double v[NV];
    for (int i = 0; i < 3; i++) v[i] = (qn[i] - qc[i]) / DT;
    {
        double ic[4], d[4], axis[3], angle, rv[3];
        qinv(qc + 3, ic); qmul(qn + 3, ic, d);
        rot_from_quat(d, axis, &angle);
        if (angle > PI) angle = angle - 2 * PI;
        if (angle < -PI) angle = angle + 2 * PI;
        for (int i = 0; i < 3; i++) rv[i] = axis[i] * angle / DT;
        // qmat(cur)^T rv, qmat normalising the quaternion
        const double *r = qc + 3;
        const double nr = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2] + r[3] * r[3]);
        const double w = r[0] / nr, x = r[1] / nr, y = r[2] / nr, z = r[3] / nr;
        const double M[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                             2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                             2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)};
        for (int i = 0; i < 3; i++) v[3 + i] = M[i] * rv[0] + M[3 + i] * rv[1] + M[6 + i] * rv[2];
    }
    for (int i = 6; i < NV; i++) v[i] = (qn[1 + i] - qc[1 + i]) / DT;
    for (int i = 0; i < NV; i++) rec[R_QVEL + i] = (Out)(v[i] < -10.0 ? -10.0 : (v[i] > 10.0 ? 10.0 : v[i]));
    for (int b = 0; b < NB; b++) {
        double ic[4], d[4], axis[3], angle;
        qinv(bc + 4 * b, ic); qmul(bn + 4 * b, ic, d);
        rot_from_quat(d, axis, &angle);
        for (int i = 0; i < 3; i++) rec[R_BANGVEL + 3 * b + i] = (Out)(axis[i] * angle / DT);
    }
    rec[R_PAD] = (Out)0; rec[R_PAD + 1] = (Out)0;
}

}  // namespace uhc_motion
