/*
 * ik_oracle.c -- CPU ORACLE (test infrastructure, NOT product code).  See ik_oracle.h.
 *
 * Every function cites the reference line it follows (paths relative to the dazzmo/ik tree) or, for
 * arithmetic that lives in the un-vendored third-party libraries, the upstream algorithm it restates
 * (Pinocchio: spatial/explog.hpp, multibody/joint/..., algorithm/{kinematics,jacobian,frames}.hxx,
 * multibody/liegroup/special-euclidean.hpp; Eigen: Cholesky/LDLT.h, Geometry/Quaternion.h).
 * Written from the published algorithms -- no third-party code is copied.  PARITY UNPINNED (header).
 */
#include <math.h>
#include <float.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* -DIKO_F32: the SAME restatement evaluated in single precision (libik_oracle_f32.so) -- what the reference computes
 * when common.hpp:13 reads `typedef float number_t` (Pinocchio and Eigen are templated on the scalar, so every
 * formula, threshold and pivot rule below is the same with Scalar = float: TaylorSeriesExpansion<float> uses
 * FLT_EPSILON).  Interface arrays become float too.  Used by tests/test_oracle_f32.py to measure how far ANY FP32
 * implementation of this iteration lands from the FP64 one (VERDICT r1 item 1c). */
#ifdef IKO_F32
#include <tgmath.h>
#define double float
#undef DBL_EPSILON
#define DBL_EPSILON FLT_EPSILON
#undef DBL_MIN
#define DBL_MIN FLT_MIN
#define IKO_TINY 1e-37f
#else
#define IKO_TINY 1e-300
#endif

#include "ik_oracle.h"

/* ------------------------------------------------------------------------------------------------
 * small helpers
 * ---------------------------------------------------------------------------------------------- */
static void cross3(const double a[3], const double b[3], double c[3]) {
    c[0] = a[1] * b[2] - a[2] * b[1];
    c[1] = a[2] * b[0] - a[0] * b[2];
    c[2] = a[0] * b[1] - a[1] * b[0];
}
static double dot3(const double a[3], const double b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
static void matvec3(const double R[9], const double v[3], double o[3]) {
    for (int i = 0; i < 3; ++i) o[i] = R[3 * i] * v[0] + R[3 * i + 1] * v[1] + R[3 * i + 2] * v[2];
}
static void matTvec3(const double R[9], const double v[3], double o[3]) {
    for (int i = 0; i < 3; ++i) o[i] = R[i] * v[0] + R[3 + i] * v[1] + R[6 + i] * v[2];
}
static void matmul3(const double A[9], const double B[9], double C[9]) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
static void matTmul3(const double A[9], const double B[9], double C[9]) { /* A^T B */
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) C[3 * i + j] = A[i] * B[j] + A[3 + i] * B[3 + j] + A[6 + i] * B[6 + j];
}

/* Pinocchio TaylorSeriesExpansion<double>::precision<degree>() = eps^(1/(degree+1)) */
static double taylor_precision(int degree) { return pow(DBL_EPSILON, 1.0 / (double)(degree + 1)); }

/* SE3 composition / inverse-composition: reference frame.hpp:48,50 (oMr.act(target), oMf.actInv(oMt)) */
void iko_se3_mul(const double A[12], const double B[12], double C[12]) {
    double R[9], p[3];
    matmul3(A, B, R);
    matvec3(A, B + 9, p);
    for (int i = 0; i < 9; ++i) C[i] = R[i];
    for (int i = 0; i < 3; ++i) C[9 + i] = A[9 + i] + p[i];
}
void iko_se3_actinv(const double A[12], const double B[12], double C[12]) {
    double R[9], d[3], p[3];
    matTmul3(A, B, R);
    for (int i = 0; i < 3; ++i) d[i] = B[9 + i] - A[9 + i];
    matTvec3(A, d, p);
    for (int i = 0; i < 9; ++i) C[i] = R[i];
    for (int i = 0; i < 3; ++i) C[9 + i] = p[i];
}

/* Eigen QuaternionBase::toRotationMatrix (used by JointModelFreeFlyer::calc); no normalisation. */
void iko_quat_to_rot(const double q[4], double R[9]) {
    const double x = q[0], y = q[1], z = q[2], w = q[3];
    const double tx = 2 * x, ty = 2 * y, tz = 2 * z;
    const double twx = tx * w, twy = ty * w, twz = tz * w;
    const double txx = tx * x, txy = ty * x, txz = tz * x;
    const double tyy = ty * y, tyz = tz * y, tzz = tz * z;
    R[0] = 1 - (tyy + tzz); R[1] = txy - twz;       R[2] = txz + twy;
    R[3] = txy + twz;       R[4] = 1 - (txx + tzz); R[5] = tyz - twx;
    R[6] = txz - twy;       R[7] = tyz + twx;       R[8] = 1 - (txx + tyy);
}

/* Eigen rotation-matrix -> quaternion assignment (quaternion::assignQuaternion in Pinocchio). */
void iko_rot_to_quat(const double R[9], double q[4]) {
    double t = R[0] + R[4] + R[8];
    if (t > 0) {
        t = sqrt(t + 1.0);
        q[3] = 0.5 * t;
        t = 0.5 / t;
        q[0] = (R[7] - R[5]) * t;
        q[1] = (R[2] - R[6]) * t;
        q[2] = (R[3] - R[1]) * t;
    } else {
        int i = 0;
        if (R[4] > R[0]) i = 1;
        if (R[8] > R[4 * i]) i = 2;
        int j = (i + 1) % 3, k = (j + 1) % 3;
        t = sqrt(R[4 * i] - R[4 * j] - R[4 * k] + 1.0);
        q[i] = 0.5 * t;
        t = 0.5 / t;
        q[3] = (R[3 * k + j] - R[3 * j + k]) * t;
        q[j] = (R[3 * j + i] + R[3 * i + j]) * t;
        q[k] = (R[3 * k + i] + R[3 * i + k]) * t;
    }
}

/* ------------------------------------------------------------------------------------------------
 * exp / log maps (Pinocchio spatial/explog.hpp restated; formulas in SURVEY.md 8c.3,4,6)
 * ---------------------------------------------------------------------------------------------- */
void iko_exp3(const double w[3], double R[9]) {
    const double t2 = dot3(w, w), t = sqrt(t2);
    double a1, a2, ct;
    if (t < taylor_precision(3)) {
        a1 = 1 - t2 / 6;
        a2 = 0.5 - t2 / 24;
        ct = 1 - t2 / 2;
    } else {
        a1 = sin(t) / t;
        a2 = (1 - cos(t)) / t2;
        ct = cos(t);
    }
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) R[3 * i + j] = a2 * w[i] * w[j];
    R[1] -= a1 * w[2]; R[3] += a1 * w[2];
    R[2] += a1 * w[1]; R[6] -= a1 * w[1];
    R[5] -= a1 * w[0]; R[7] += a1 * w[0];
    R[0] += ct; R[4] += ct; R[8] += ct;
}

void iko_exp6(const double nu[6], double M[12]) {
    const double *v = nu, *w = nu + 3;
    const double t2 = dot3(w, w), t = sqrt(t2);
    double alpha_wxv, alpha_v, alpha_w, diag;
    if (t < taylor_precision(3)) {
        alpha_wxv = 0.5 - t2 / 24;
        alpha_v = 1 - t2 / 6;
        alpha_w = 1.0 / 6 - t2 / 120;
        diag = 1 - t2 / 2;
    } else {
        const double st = sin(t), ct = cos(t), inv_t2 = 1 / t2;
        alpha_wxv = (1 - ct) * inv_t2;
        alpha_v = st / t;
        alpha_w = (1 - alpha_v) * inv_t2;
        diag = ct;
    }
    double wxv[3];
    cross3(w, v, wxv);
    const double wv = dot3(w, v);
    for (int i = 0; i < 3; ++i) M[9 + i] = alpha_v * v[i] + (alpha_w * wv) * w[i] + alpha_wxv * wxv[i];
    double *R = M;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) R[3 * i + j] = alpha_wxv * w[i] * w[j];
    R[1] -= alpha_v * w[2]; R[3] += alpha_v * w[2];
    R[2] += alpha_v * w[1]; R[6] -= alpha_v * w[1];
    R[5] -= alpha_v * w[0]; R[7] += alpha_v * w[0];
    R[0] += diag; R[4] += diag; R[8] += diag;
}

void iko_log3(const double R[9], double w[3], double *theta) {
    const double PI_ = 3.14159265358979323846;
    const double tr = R[0] + R[4] + R[8];
    double t;
    if (tr >= 3.0) t = 0.0;
    else if (tr <= -1.0) t = PI_;
    else t = acos((tr - 1) / 2);
    if (t >= PI_ - 1e-2) {
        /* near pi: diagonal-based formula (precision sqrt of the antisymmetric one) */
        const double cphi = -(tr - 1) / 2;
        const double beta = t * t / (1 + cphi);
        const double d0 = (R[0] + cphi) * beta, d1 = (R[4] + cphi) * beta, d2 = (R[8] + cphi) * beta;
        w[0] = (R[7] > R[5] ? 1.0 : -1.0) * (d0 > 0 ? sqrt(d0) : 0.0);
        w[1] = (R[2] > R[6] ? 1.0 : -1.0) * (d1 > 0 ? sqrt(d1) : 0.0);
        w[2] = (R[3] > R[1] ? 1.0 : -1.0) * (d2 > 0 ? sqrt(d2) : 0.0);
    } else {
        const double s = (t > taylor_precision(2) ? t / sin(t) : 1.0) / 2;
        w[0] = s * (R[7] - R[5]);
        w[1] = s * (R[2] - R[6]);
        w[2] = s * (R[3] - R[1]);
    }
    *theta = t;
}

void iko_log6(const double M[12], double out[6]) {
    const double *p = M + 9;
    double w[3], t;
    iko_log3(M, w, &t);
    const double t2 = t * t;
    double alpha, beta;
    if (t < taylor_precision(3)) {
        alpha = 1 - t2 / 12 - t2 * t2 / 720;
        beta = 1.0 / 12 + t2 / 720;
    } else {
        const double st = sin(t), ct = cos(t);
        alpha = t * st / (2 * (1 - ct));
        beta = 1 / t2 - st / (2 * t * (1 - ct));
    }
    double wxp[3];
    cross3(w, p, wxp);
    const double wp = dot3(w, p);
    for (int i = 0; i < 3; ++i) {
        out[i] = alpha * p[i] - 0.5 * wxp[i] + (beta * wp) * w[i];
        out[3 + i] = w[i];
    }
}

static void add_skew(const double v[3], double s, double M[9]) {
    M[1] -= s * v[2]; M[2] += s * v[1];
    M[3] += s * v[2]; M[5] -= s * v[0];
    M[6] -= s * v[1]; M[7] += s * v[0];
}

void iko_Jlog3(double t, const double w[3], double J[9]) {
    double alpha, diag;
    if (t < taylor_precision(3)) {
        alpha = 1.0 / 12 + t * t / 720;
        diag = 0.5 * (2 - t * t / 6);
    } else {
        const double st = sin(t), ct = cos(t);
        const double st_1mct = st / (1 - ct);
        alpha = 1 / (t * t) - st_1mct / (2 * t);
        diag = 0.5 * (t * st_1mct);
    }
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) J[3 * i + j] = alpha * w[i] * w[j];
    J[0] += diag; J[4] += diag; J[8] += diag;
    add_skew(w, 0.5, J);
}

/* Jlog6(M) = [[A, B], [0, A]], row-major 6x6; log6(M*exp6(xi)) ~ log6(M) + Jlog6(M) xi. */
void iko_Jlog6(const double M[12], double J[36]) {
    const double *p = M + 9;
    double w[3], t, A[9], C[9], B[9];
    iko_log3(M, w, &t);
    iko_Jlog3(t, w, A);
    const double t2 = t * t;
    double beta, bdot;
    if (t < taylor_precision(3)) {
        beta = 1.0 / 12 + t2 / 720;
        bdot = 1.0 / 360;
    } else {
        const double tinv = 1 / t, t2inv = tinv * tinv;
        const double st = sin(t), ct = cos(t);
        const double inv_2_2ct = 1 / (2 * (1 - ct));
        beta = t2inv - st * tinv * inv_2_2ct;
        bdot = -2 * t2inv * t2inv + (1 + st * tinv) * t2inv * inv_2_2ct;
    }
    const double wTp = dot3(w, p);
    double v3[3];
    for (int i = 0; i < 3; ++i) v3[i] = (bdot * wTp) * w[i] - (t2 * bdot + 2 * beta) * p[i];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) C[3 * i + j] = v3[i] * w[j] + beta * w[i] * p[j];
    C[0] += wTp * beta; C[4] += wTp * beta; C[8] += wTp * beta;
    add_skew(p, 0.5, C);
    matmul3(C, A, B);
    memset(J, 0, 36 * sizeof(double));
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            J[6 * i + j] = A[3 * i + j];
            J[6 * i + 3 + j] = B[3 * i + j];
            J[6 * (3 + i) + 3 + j] = A[3 * i + j];
        }
}

/* ------------------------------------------------------------------------------------------------
 * kinematics
 * ---------------------------------------------------------------------------------------------- */
static void joint_axis(const iko_model *m, int j, double a[3]) {
    a[0] = a[1] = a[2] = 0.0;
    switch (m->jtype[j]) {
        case IKO_J_RX: case IKO_J_PX: a[0] = 1; break;
        case IKO_J_RY: case IKO_J_PY: a[1] = 1; break;
        case IKO_J_RZ: case IKO_J_PZ: a[2] = 1; break;
        default: a[0] = m->axis[3 * j]; a[1] = m->axis[3 * j + 1]; a[2] = m->axis[3 * j + 2];
    }
}

/* joint transform M_j(q) (Pinocchio Joint*::calc) */
static void joint_transform(const iko_model *m, int j, const double *q, double M[12]) {
    const int t = m->jtype[j];
    const double *qj = q + m->idx_q[j];
    for (int i = 0; i < 12; ++i) M[i] = 0;
    M[0] = M[4] = M[8] = 1;
    if (t == IKO_J_FREEFLYER) {
        iko_quat_to_rot(qj + 3, M);
        M[9] = qj[0]; M[10] = qj[1]; M[11] = qj[2];
    } else if (t >= IKO_J_RX && t <= IKO_J_REV_UNALIGNED) {
        const double s = sin(qj[0]), c = cos(qj[0]);
        if (t == IKO_J_RX) { M[4] = c; M[5] = -s; M[7] = s; M[8] = c; }
        else if (t == IKO_J_RY) { M[0] = c; M[2] = s; M[6] = -s; M[8] = c; }
        else if (t == IKO_J_RZ) { M[0] = c; M[1] = -s; M[3] = s; M[4] = c; }
        else { /* Rodrigues about a unit axis */
            double a[3];
            joint_axis(m, j, a);
            const double v = 1 - c;
            M[0] = a[0] * a[0] * v + c;        M[1] = a[0] * a[1] * v - a[2] * s; M[2] = a[0] * a[2] * v + a[1] * s;
            M[3] = a[0] * a[1] * v + a[2] * s; M[4] = a[1] * a[1] * v + c;        M[5] = a[1] * a[2] * v - a[0] * s;
            M[6] = a[0] * a[2] * v - a[1] * s; M[7] = a[1] * a[2] * v + a[0] * s; M[8] = a[2] * a[2] * v + c;
        }
    } else if (t >= IKO_J_PX && t <= IKO_J_PRIS_UNALIGNED) {
        double a[3];
        joint_axis(m, j, a);
        M[9] = a[0] * qj[0]; M[10] = a[1] * qj[0]; M[11] = a[2] * qj[0];
    }
}

/* pinocchio::forwardKinematics part of framesForwardKinematics (reference data.cpp:28-29):
 * liMi = placement * M_j(q); oMi = oMi[parent] * liMi. */
void iko_fk(const iko_model *m, const double *q, double *oMi) {
    for (int i = 0; i < 12; ++i) oMi[i] = 0;
    oMi[0] = oMi[4] = oMi[8] = 1;
    for (int j = 1; j < m->njoints; ++j) {
        double Mj[12], li[12];
        joint_transform(m, j, q, Mj);
        iko_se3_mul(m->placement + 12 * j, Mj, li);
        if (m->parent[j] > 0) iko_se3_mul(oMi + 12 * m->parent[j], li, oMi + 12 * j);
        else memcpy(oMi + 12 * j, li, sizeof(li));
    }
}

/* updateFramePlacements: oMf = oMi[parent] * placement_f (reference common.hpp:47-51 reads it) */
void iko_frame_placement(const iko_model *m, const double *oMi, int f, double oMf[12]) {
    iko_se3_mul(oMi + 12 * m->frame_parent[f], m->frame_placement + 12 * f, oMf);
}

/* pinocchio::computeJointJacobians (reference data.cpp:30): world columns oMi.act(S_i). */
void iko_joint_jacobians(const iko_model *m, const double *oMi, double *J) {
    const int nv = m->nv;
    memset(J, 0, sizeof(double) * 6 * nv);
    for (int j = 1; j < m->njoints; ++j) {
        const double *R = oMi + 12 * j, *p = R + 9;
        const int c0 = m->idx_v[j], t = m->jtype[j];
        if (t == IKO_J_FREEFLYER) {
            /* action matrix [[R, p^ R], [0, R]] */
            for (int c = 0; c < 3; ++c) {
                double rc[3] = {R[c], R[3 + c], R[6 + c]}, pxr[3];
                cross3(p, rc, pxr);
                for (int r = 0; r < 3; ++r) {
                    J[r * nv + c0 + c] = rc[r];
                    J[r * nv + c0 + 3 + c] = pxr[r];
                    J[(3 + r) * nv + c0 + 3 + c] = rc[r];
                }
            }
        } else if (t >= IKO_J_RX && t <= IKO_J_REV_UNALIGNED) {
            double a[3], z[3], pxz[3];
            joint_axis(m, j, a);
            matvec3(R, a, z);
            cross3(p, z, pxz);
            for (int r = 0; r < 3; ++r) { J[r * nv + c0] = pxz[r]; J[(3 + r) * nv + c0] = z[r]; }
        } else if (t >= IKO_J_PX && t <= IKO_J_PRIS_UNALIGNED) {
            double a[3], z[3];
            joint_axis(m, j, a);
            matvec3(R, a, z);
            for (int r = 0; r < 3; ++r) J[r * nv + c0] = z[r];
        }
    }
}

static int joint_nv(const iko_model *m, int j) { return m->jtype[j] == IKO_J_FREEFLYER ? 6 : (m->jtype[j] == IKO_J_UNIVERSE ? 0 : 1); }

/* pinocchio::getFrameJacobian(model, data, id, LOCAL, J) (reference frame.hpp:169-170): for every
 * joint supporting the frame, J.col = oMf.actInv(data.J.col); other columns are left untouched (zero). */
void iko_frame_jacobian_local(const iko_model *m, const double *oMi, const double *Jw, int f, double *Jf) {
    const int nv = m->nv;
    double oMf[12];
    iko_frame_placement(m, oMi, f, oMf);
    memset(Jf, 0, sizeof(double) * 6 * nv);
    for (int j = m->frame_parent[f]; j > 0; j = m->parent[j]) {
        for (int c = m->idx_v[j]; c < m->idx_v[j] + joint_nv(m, j); ++c) {
            double v[3] = {Jw[c], Jw[nv + c], Jw[2 * nv + c]};
            double w[3] = {Jw[3 * nv + c], Jw[4 * nv + c], Jw[5 * nv + c]};
            double pxw[3], d[3], lv[3], lw[3];
            cross3(oMf + 9, w, pxw);
            for (int i = 0; i < 3; ++i) d[i] = v[i] - pxw[i];
            matTvec3(oMf, d, lv);
            matTvec3(oMf, w, lw);
            for (int i = 0; i < 3; ++i) { Jf[i * nv + c] = lv[i]; Jf[(3 + i) * nv + c] = lw[i]; }
        }
    }
}

/* pinocchio::integrate (reference dls.cpp:67-68).  Free-flyer: SpecialEuclideanOperation<3>::integrate_impl
 * (M1 = M0*exp6(v); quaternion from M1.rotation, sign made continuous with the old one, first-order
 * normalisation alpha = (3 - |q|^2)/2).  Revolute / prismatic: q + v. */
void iko_integrate(const iko_model *m, const double *q, const double *v, double *qout) {
    for (int j = 1; j < m->njoints; ++j) {
        const int iq = m->idx_q[j], iv = m->idx_v[j];
        if (m->jtype[j] == IKO_J_FREEFLYER) {
            double M0[12], E[12], M1[12], quat[4];
            iko_quat_to_rot(q + iq + 3, M0);
            M0[9] = q[iq]; M0[10] = q[iq + 1]; M0[11] = q[iq + 2];
            iko_exp6(v + iv, E);
            iko_se3_mul(M0, E, M1);
            qout[iq] = M1[9]; qout[iq + 1] = M1[10]; qout[iq + 2] = M1[11];
            iko_rot_to_quat(M1, quat);
            double dotp = 0;
            for (int i = 0; i < 4; ++i) dotp += quat[i] * q[iq + 3 + i];
            if (dotp < 0) for (int i = 0; i < 4; ++i) quat[i] = -quat[i];
            double n2 = 0;
            for (int i = 0; i < 4; ++i) n2 += quat[i] * quat[i];
            const double alpha = (3 - n2) / 2;
            for (int i = 0; i < 4; ++i) qout[iq + 3 + i] = quat[i] * alpha;
        } else {
            qout[iq] = q[iq] + v[iv];
        }
    }
}

/* reference common.hpp:53-56: q = min(upper, max(q, lower)) over ALL nq entries */
void iko_clip(const iko_model *m, double *q) {
    for (int i = 0; i < m->nq; ++i) {
        double x = q[i] > m->lower[i] ? q[i] : m->lower[i]; /* cwiseMax(lower) */
        q[i] = m->upper[i] < x ? m->upper[i] : x;           /* upper.cwiseMin(.) */
    }
}

/* ------------------------------------------------------------------------------------------------
 * problem bookkeeping (reference problem.hpp:34-40, frame.hpp:100-107, posture.hpp:27-33)
 * ---------------------------------------------------------------------------------------------- */
/* pinocchio::jacobianCenterOfMass(model, data, q, false) (data.cpp:31-34): backward pass over the tree accumulating the
 * mass and first moment of every subtree; the column of a joint coordinate is the velocity it gives its subtree's centre
 * of mass, scaled by the subtree's share of the total mass.  Bodies attached to `universe` are not counted (Pinocchio's
 * loops start at joint 1). */
void iko_center_of_mass(const iko_model *m, const double *q, double com[3], double *Jcom) {
    const int nj = m->njoints, nv = m->nv;
    double *oMi = (double *)malloc(sizeof(double) * 12 * nj), *Jw = (double *)malloc(sizeof(double) * 6 * nv);
    double *ms = (double *)calloc(nj, sizeof(double)), *mc = (double *)calloc(3 * nj, sizeof(double));
    iko_fk(m, q, oMi);
    iko_joint_jacobians(m, oMi, Jw);
    for (int j = 1; j < nj; ++j) {
        double cw[3];
        matvec3(oMi + 12 * j, m->com + 3 * j, cw);
        ms[j] = m->mass[j];
        for (int i = 0; i < 3; ++i) mc[3 * j + i] = m->mass[j] * (cw[i] + oMi[12 * j + 9 + i]);
    }
    double M = 0, tot[3] = {0, 0, 0};
    for (int j = nj - 1; j >= 1; --j) {
        const int p = m->parent[j];
        if (p > 0) {
            ms[p] += ms[j];
            for (int i = 0; i < 3; ++i) mc[3 * p + i] += mc[3 * j + i];
        } else {
            M += ms[j];
            for (int i = 0; i < 3; ++i) tot[i] += mc[3 * j + i];
        }
    }
    for (int i = 0; i < 3; ++i) com[i] = tot[i] / M;
    if (Jcom) {
        memset(Jcom, 0, sizeof(double) * 3 * nv);
        for (int j = 1; j < nj; ++j) {
            if (!(ms[j] > 0)) continue;
            const double cs[3] = {mc[3 * j] / ms[j], mc[3 * j + 1] / ms[j], mc[3 * j + 2] / ms[j]};
            for (int c = m->idx_v[j]; c < m->idx_v[j] + joint_nv(m, j); ++c) {
                const double v[3] = {Jw[c], Jw[nv + c], Jw[2 * nv + c]}, w[3] = {Jw[3 * nv + c], Jw[4 * nv + c], Jw[5 * nv + c]};
                double wxc[3];
                cross3(w, cs, wxc);
                for (int i = 0; i < 3; ++i) Jcom[i * nv + c] = ms[j] / M * (v[i] + wxc[i]);
            }
        }
    }
    free(oMi); free(Jw); free(ms); free(mc);
}

int iko_task_dim(const iko_problem *pb, int t) {
    if (pb->kind[t] == IKO_TASK_FRAME) return pb->type[t] == IKO_FULL ? 6 : 3;
    if (pb->kind[t] == IKO_TASK_ALIGN_AXIS) return 1;
    if (pb->kind[t] == IKO_TASK_COM) return 3;
    return pb->type[t]; /* posture: nj */
}
int iko_task_target_size(const iko_problem *pb, int t) {
    if (pb->kind[t] == IKO_TASK_FRAME) return 12;
    if (pb->kind[t] == IKO_TASK_ALIGN_AXIS) return 3;
    if (pb->kind[t] == IKO_TASK_COM) return 3;
    return pb->type[t];
}
int iko_target_size(const iko_problem *pb) {
    int s = 0;
    for (int t = 0; t < pb->ntasks; ++t) s += iko_task_target_size(pb, t);
    return s;
}
int iko_e_size(const iko_problem *pb, int priority) {
    int s = 0;
    for (int t = 0; t < pb->ntasks; ++t)
        if (pb->priority[t] == priority) s += iko_task_dim(pb, t);
    return s;
}
int iko_total_rows(const iko_problem *pb) {
    int s = 0;
    for (int t = 0; t < pb->ntasks; ++t) s += iko_task_dim(pb, t);
    return s;
}

/* evaluate_problem_data (reference data.cpp:25-58) followed by the stacking of dls.cpp:18-24:
 * rows ordered by priority level, then by insertion order inside the level. */
void iko_evaluate(const iko_model *m, const iko_problem *pb, const double *q, const double *targets, double *e,
                  double *J) {
    const int nv = m->nv, rows = iko_total_rows(pb);
    double *oMi = (double *)malloc(sizeof(double) * 12 * m->njoints);
    double *Jw = (double *)malloc(sizeof(double) * 6 * nv);
    double *Jf = (double *)malloc(sizeof(double) * 6 * nv);
    iko_fk(m, q, oMi);                 /* data.cpp:28-29 */
    iko_joint_jacobians(m, oMi, Jw);   /* data.cpp:30 */
    memset(J, 0, sizeof(double) * rows * nv);

    int row = 0;
    for (int p = 0; p <= pb->max_priority_level; ++p) {
        int toff = 0, woff = 0, moff = 0;
        for (int t = 0; t < pb->ntasks; ++t) {
            const int dim = iko_task_dim(pb, t), tsz = iko_task_target_size(pb, t);
            if (pb->priority[t] == p) {
                const double *tg = targets + toff;
                double *et = e + row, *Jt = J + row * nv;
                if (pb->kind[t] == IKO_TASK_FRAME) {
                    /* compute_frame_error, frame.hpp:37-62 */
                    double oMf[12], oMr[12], oMt[12], fMt[12], tMf[12], lg[6], Jl[36];
                    iko_frame_placement(m, oMi, pb->frame[t], oMf);
                    iko_frame_placement(m, oMi, pb->ref[t], oMr);
                    iko_se3_mul(oMr, tg, oMt);
                    iko_se3_actinv(oMf, oMt, fMt);
                    iko_log6(fMt, lg);
                    const int r0 = pb->type[t] == IKO_ORIENTATION ? 3 : 0;
                    for (int i = 0; i < dim; ++i) et[i] = lg[r0 + i];
                    /* FrameTask::compute_jacobian, frame.hpp:152-182: J = rows of (-Jlog6(tMf) * Jf_LOCAL) */
                    iko_se3_actinv(oMt, oMf, tMf);
                    iko_Jlog6(tMf, Jl);
                    iko_frame_jacobian_local(m, oMi, Jw, pb->frame[t], Jf);
                    for (int i = 0; i < dim; ++i)
                        for (int c = 0; c < nv; ++c) {
                            double s = 0;
                            for (int k = 0; k < 6; ++k) s += -Jl[6 * (r0 + i) + k] * Jf[k * nv + c];
                            Jt[i * nv + c] = s;
                        }
                } else if (pb->kind[t] == IKO_TASK_ALIGN_AXIS) {
                    /* AlignAxisTask, frame.hpp:246-299: e = 1 - r.t^, J = -(r x t^)^T R_rMf Jf_angular */
                    double oMf[12], oMr[12], rMf[12];
                    iko_frame_placement(m, oMi, pb->frame[t], oMf);
                    iko_frame_placement(m, oMi, pb->ref[t], oMr);
                    iko_se3_actinv(oMr, oMf, rMf);
                    const int ax = pb->type[t];
                    double r[3] = {rMf[ax], rMf[3 + ax], rMf[6 + ax]};
                    const double n = sqrt(dot3(tg, tg));
                    double tn[3] = {tg[0] / n, tg[1] / n, tg[2] / n}, rxt[3], row3[3];
                    et[0] = 1.0 - dot3(r, tn);
                    cross3(r, tn, rxt);
                    matTvec3(rMf, rxt, row3); /* (r x t)^T R */
                    iko_frame_jacobian_local(m, oMi, Jw, pb->frame[t], Jf);
                    for (int c = 0; c < nv; ++c)
                        Jt[c] = -(row3[0] * Jf[3 * nv + c] + row3[1] * Jf[4 * nv + c] + row3[2] * Jf[5 * nv + c]);
                } else if (pb->kind[t] == IKO_TASK_COM) {
                    /* CentreOfMassTask, centre_of_mass.hpp:24-38: e = oMr^-1 com - target; J = R_r^T Jcom (the reference frame
                     * is not differentiated, like everywhere else in the reference) */
                    double com[3], oMr[12], d[3];
                    double *Jcom = (double *)malloc(sizeof(double) * 3 * nv);
                    iko_center_of_mass(m, q, com, Jcom);
                    iko_frame_placement(m, oMi, pb->ref[t], oMr);
                    for (int i = 0; i < 3; ++i) d[i] = com[i] - oMr[9 + i];
                    matTvec3(oMr, d, et);
                    for (int i = 0; i < 3; ++i) et[i] -= tg[i];
                    for (int c = 0; c < nv; ++c) {
                        double col[3] = {Jcom[c], Jcom[nv + c], Jcom[2 * nv + c]}, lc[3];
                        matTvec3(oMr, col, lc);
                        for (int i = 0; i < 3; ++i) Jt[i * nv + c] = lc[i];
                    }
                    free(Jcom);
                } else {
                    /* PostureTask, posture.hpp:50-67: e = (q.tail(nj) - target) o mask; J.rightCols(nj) = I */
                    const int nj = pb->type[t];
                    for (int i = 0; i < nj; ++i) {
                        et[i] = (q[m->nq - nj + i] - tg[i]) * pb->mask[moff + i];
                        Jt[i * nv + (nv - nj + i)] = 1.0;
                    }
                }
                /* weighting, data.cpp:49-50 */
                for (int i = 0; i < dim; ++i) {
                    et[i] *= pb->weight[woff + i];
                    for (int c = 0; c < nv; ++c) Jt[i * nv + c] *= pb->weight[woff + i];
                }
                row += dim;
            }
            toff += tsz;
            woff += dim;
            if (pb->kind[t] == IKO_TASK_POSTURE) moff += pb->type[t];
        }
    }
    free(oMi); free(Jw); free(Jf);
}

/* ------------------------------------------------------------------------------------------------
 * Eigen::LDLT restated (Cholesky/LDLT.h: ldlt_inplace<Lower>::unblocked + _solve_impl): symmetric
 * pivoting on the largest remaining diagonal entry, A = P^T L D L^T P; solve uses D's pseudo-inverse.
 * Reference call site: dls.cpp:53  data.JJ.ldlt().solve(data.et).
 * ---------------------------------------------------------------------------------------------- */
int iko_c_size(const iko_problem *pb) {
    int n = 0;
    for (int k = 0; k < pb->nconstraints; ++k) n += pb->c_type[k] == IKO_FULL ? 6 : 3;
    return n;
}

/* FrameConstraint::compute_jacobian (frame.hpp:399-437) for every constraint, stacked in insertion order (dls.cpp:26-34) */
void iko_constraint_jacobian(const iko_model *m, const iko_problem *pb, const double *q, double *Jc) {
    const int nv = m->nv;
    double *oMi = (double *)malloc(sizeof(double) * 12 * m->njoints);
    double *Jw = (double *)malloc(sizeof(double) * 6 * nv);
    double *Jf = (double *)malloc(sizeof(double) * 6 * nv), *Jr = (double *)malloc(sizeof(double) * 6 * nv);
    iko_fk(m, q, oMi);
    iko_joint_jacobians(m, oMi, Jw);
    int row = 0;
    for (int k = 0; k < pb->nconstraints; ++k) {
        double oMf[12], oMr[12], rMf[12];
        iko_frame_placement(m, oMi, pb->c_frame[k], oMf);
        iko_frame_placement(m, oMi, pb->c_ref[k], oMr);
        iko_se3_actinv(oMr, oMf, rMf);                                      /* frame.hpp:407 */
        iko_frame_jacobian_local(m, oMi, Jw, pb->c_frame[k], Jf);           /* frame.hpp:410-411 */
        iko_frame_jacobian_local(m, oMi, Jw, pb->c_ref[k], Jr);             /* frame.hpp:414-416 */
        /* rMf.toActionMatrixInverse() = [[R^T, -R^T p^], [0, R^T]] for rMf = (R, p): (v, w) -> (R^T (v - p x w), R^T w) */
        const double *R = rMf, *p = rMf + 9;
        const int full = pb->c_type[k] == IKO_FULL, r0 = pb->c_type[k] == IKO_ORIENTATION ? 3 : 0, dim = full ? 6 : 3;
        for (int c = 0; c < nv; ++c) {
            double v[3] = {Jr[c], Jr[nv + c], Jr[2 * nv + c]}, w[3] = {Jr[3 * nv + c], Jr[4 * nv + c], Jr[5 * nv + c]};
            double pxw[3], d[3], lv[3], lw[3], col[6];
            cross3(p, w, pxw);
            for (int i = 0; i < 3; ++i) d[i] = v[i] - pxw[i];
            matTvec3(R, d, lv);
            matTvec3(R, w, lw);
            for (int i = 0; i < 3; ++i) { col[i] = Jf[i * nv + c] - lv[i]; col[3 + i] = Jf[(3 + i) * nv + c] - lw[i]; }
            for (int i = 0; i < dim; ++i) Jc[(row + i) * nv + c] = col[r0 + i];     /* frame.hpp:420-436 */
        }
        row += dim;
    }
    free(oMi); free(Jw); free(Jf); free(Jr);
}

void iko_ldlt_solve(int n, double *A, const double *b, double *x) {
    int *tr = (int *)malloc(sizeof(int) * (n > 0 ? n : 1));
    double *tmp = (double *)malloc(sizeof(double) * (n > 0 ? n : 1));
#define a_(i, j) A[(i) * n + (j)]
    for (int k = 0; k < n; ++k) {
        int big = k;
        double bv = fabs(a_(k, k));
        for (int i = k + 1; i < n; ++i)
            if (fabs(a_(i, i)) > bv) { bv = fabs(a_(i, i)); big = i; }
        tr[k] = big;
        if (big != k) { /* symmetric swap touching only the lower triangle */
            for (int j = 0; j < k; ++j) { double t = a_(k, j); a_(k, j) = a_(big, j); a_(big, j) = t; }
            for (int i = big + 1; i < n; ++i) { double t = a_(i, k); a_(i, k) = a_(i, big); a_(i, big) = t; }
            { double t = a_(k, k); a_(k, k) = a_(big, big); a_(big, big) = t; }
            for (int i = k + 1; i < big; ++i) { double t = a_(i, k); a_(i, k) = a_(big, i); a_(big, i) = t; }
        }
        if (k > 0) {
            for (int j = 0; j < k; ++j) tmp[j] = a_(j, j) * a_(k, j);
            double s = 0;
            for (int j = 0; j < k; ++j) s += a_(k, j) * tmp[j];
            a_(k, k) -= s;
            for (int i = k + 1; i < n; ++i) {
                double u = 0;
                for (int j = 0; j < k; ++j) u += a_(i, j) * tmp[j];
                a_(i, k) -= u;
            }
        }
        const double akk = a_(k, k);
        if (fabs(akk) > 0)
            for (int i = k + 1; i < n; ++i) a_(i, k) /= akk;
    }
    for (int i = 0; i < n; ++i) x[i] = b[i];
    for (int k = 0; k < n; ++k) { double t = x[k]; x[k] = x[tr[k]]; x[tr[k]] = t; }        /* P b */
    for (int i = 0; i < n; ++i) for (int j = 0; j < i; ++j) x[i] -= a_(i, j) * x[j];       /* L^-1 */
    for (int i = 0; i < n; ++i) x[i] = fabs(a_(i, i)) > DBL_MIN ? x[i] / a_(i, i) : 0.0;   /* D^+  */
    for (int i = n - 1; i >= 0; --i) for (int j = i + 1; j < n; ++j) x[i] -= a_(j, i) * x[j]; /* L^-T */
    for (int k = n - 1; k >= 0; --k) { double t = x[k]; x[k] = x[tr[k]]; x[tr[k]] = t; }   /* P^T */
#undef a_
    free(tr); free(tmp);
}

/* ------------------------------------------------------------------------------------------------
 * ik::dls, reference dls.cpp:5-78 (no constraints: N = I, dls.cpp:44-45)
 * ---------------------------------------------------------------------------------------------- */
int iko_dls(const iko_model *m, const iko_problem *pb, const iko_params *prm, const double *q0, const double *targets,
            double *q_out, int *iters, double *resid, double *dq_out) {
    const int nq = m->nq, nv = m->nv, rows = iko_total_rows(pb), r0 = iko_e_size(pb, 0);
    double *q = (double *)malloc(sizeof(double) * nq), *qn = (double *)malloc(sizeof(double) * nq);
    double *e = (double *)malloc(sizeof(double) * (rows + 1)), *J = (double *)malloc(sizeof(double) * (rows * nv + 1));
    double *JJ = (double *)malloc(sizeof(double) * (rows * rows + 1)), *y = (double *)malloc(sizeof(double) * (rows + 1));
    double *dq = (double *)malloc(sizeof(double) * nv), *sdq = (double *)malloc(sizeof(double) * nv);
    memcpy(q, q0, sizeof(double) * nq);                                     /* dls.cpp:8 */
    int success = 0, it = 0;
    double res = 0;
    const int crows = iko_c_size(pb);
    double *Jc = (double *)malloc(sizeof(double) * (crows * nv + 1)), *N = (double *)malloc(sizeof(double) * nv * nv);
    for (it = 0; it < prm->max_iterations; ++it) {                           /* dls.cpp:14 */
        iko_evaluate(m, pb, q, targets, e, J);                               /* dls.cpp:16-24 */
        for (int i = 0; i < rows; ++i)                                       /* dls.cpp:39 */
            for (int j = 0; j < rows; ++j) {
                double s = 0;
                for (int c = 0; c < nv; ++c) s += J[i * nv + c] * J[j * nv + c];
                JJ[i * rows + j] = s;
            }
        for (int i = 0; i < rows; ++i) JJ[i * rows + i] += prm->damping * prm->damping; /* dls.cpp:41 */
        iko_ldlt_solve(rows, JJ, e, y);                                      /* dls.cpp:53 */
        for (int c = 0; c < nv; ++c) {                                       /* dls.cpp:52 */
            double s = 0;
            for (int i = 0; i < rows; ++i) s += J[i * nv + c] * y[i];
            dq[c] = -s;
        }
        if (crows > 0) {                                                     /* dls.cpp:26-34,44-52: dq = -N (J^T y) */
            iko_constraint_jacobian(m, pb, q, Jc);
            iko_rowspace_projector(crows, nv, Jc, N);                        /* Jc.cod().pseudoInverse() * Jc */
            for (int c = 0; c < nv; ++c) {
                double s = 0;
                for (int k = 0; k < nv; ++k) s += N[c * nv + k] * dq[k];
                sdq[c] = dq[c] - s;                                          /* (I - Jc^+ Jc) dq */
            }
            memcpy(dq, sdq, sizeof(double) * nv);
        }
        res = 0;                                                             /* visitor.hpp:19 */
        for (int i = 0; i < r0; ++i) res += e[i] * e[i];
        if (res < prm->tolerance) { success = 1; break; }                    /* dls.cpp:61-64 */
        for (int c = 0; c < nv; ++c) sdq[c] = prm->step_length * dq[c];
        iko_integrate(m, q, sdq, qn);                                        /* dls.cpp:67-68 */
        memcpy(q, qn, sizeof(double) * nq);
        iko_clip(m, q);                                                      /* dls.cpp:71 */
    }
    memcpy(q_out, q, sizeof(double) * nq);                                   /* dls.cpp:63 / 77 */
    if (iters) *iters = it;
    if (resid) *resid = res;
    if (dq_out) memcpy(dq_out, dq, sizeof(double) * nv);
    free(q); free(qn); free(e); free(J); free(JJ); free(y); free(dq); free(sdq); free(Jc); free(N);
    return success;
}

typedef struct {
    const iko_model *m; const iko_problem *pb; const iko_params *prm;
    int b0, b1;
    const double *q0, *targets;
    double *q_out; unsigned char *success; int *iters; double *resid;
} batch_job;

static void *batch_worker(void *arg) {
    batch_job *j = (batch_job *)arg;
    const int nq = j->m->nq, tsz = iko_target_size(j->pb);
    for (int b = j->b0; b < j->b1; ++b) {
        int it; double r;
        int ok = iko_dls(j->m, j->pb, j->prm, j->q0 + (size_t)b * nq, j->targets + (size_t)b * tsz,
                         j->q_out + (size_t)b * nq, &it, &r, 0);
        j->success[b] = (unsigned char)ok;
        if (j->iters) j->iters[b] = it;
        if (j->resid) j->resid[b] = r;
    }
    return 0;
}

void iko_dls_batch(const iko_model *m, const iko_problem *pb, const iko_params *prm, int B, const double *q0,
                   const double *targets, double *q_out, unsigned char *success, int *iters, double *resid,
                   int nthreads) {
    if (nthreads < 1) nthreads = 1;
    if (nthreads > B) nthreads = B > 0 ? B : 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * nthreads);
    batch_job *jobs = (batch_job *)malloc(sizeof(batch_job) * nthreads);
    for (int t = 0; t < nthreads; ++t) {
        batch_job jb = {m, pb, prm, (int)((long long)B * t / nthreads), (int)((long long)B * (t + 1) / nthreads),
                        q0, targets, q_out, success, iters, resid};
        jobs[t] = jb;
        if (nthreads == 1) batch_worker(&jobs[t]);
        else pthread_create(&th[t], 0, batch_worker, &jobs[t]);
    }
    if (nthreads > 1)
        for (int t = 0; t < nthreads; ++t) pthread_join(th[t], 0);
    free(th); free(jobs);
}

/* ======================================================================================================
 * ik::pik -- priority-based IK (reference ik/ik/pik.cpp:5-96, pik.hpp:13-57).  SURVEY 8f rank 2.
 * ====================================================================================================== */

/* Thin SVD of A (m x n, row-major, m <= n) by one-sided Jacobi on the rows: A = U diag(s) V^T with U m x m, V n x m.
 * (Eigen::JacobiSVD, pik.cpp:8-9, is a two-sided Jacobi; singular triplets are unique up to sign / order for distinct
 * values, and damp_pseudoinverse sums over all of them, so any converged SVD gives the same matrix.) */
static void svd_rows(int m, int n, const double *A, double *U, double *s, double *V) {
    double *W = (double *)malloc(sizeof(double) * m * n); /* rows become s_i * v_i^T */
    memcpy(W, A, sizeof(double) * m * n);
    for (int i = 0; i < m; ++i)
        for (int j = 0; j < m; ++j) U[i * m + j] = (i == j);
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0;
        for (int p = 0; p < m - 1; ++p)
            for (int q = p + 1; q < m; ++q) {
                double a = 0, b = 0, c = 0;
                for (int k = 0; k < n; ++k) {
                    a += W[p * n + k] * W[p * n + k];
                    b += W[q * n + k] * W[q * n + k];
                    c += W[p * n + k] * W[q * n + k];
                }
                if (fabs(c) <= IKO_TINY || fabs(c) <= 1e-17 * sqrt(a * b)) continue;
                off += fabs(c) / sqrt(a * b + IKO_TINY);
                const double zeta = (b - a) / (2 * c);
                const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1 + zeta * zeta));
                const double cs = 1 / sqrt(1 + t * t), sn = cs * t;
                for (int k = 0; k < n; ++k) {
                    const double wp = W[p * n + k], wq = W[q * n + k];
                    W[p * n + k] = cs * wp - sn * wq;
                    W[q * n + k] = sn * wp + cs * wq;
                }
                for (int k = 0; k < m; ++k) { /* A = U W: rows of W rotated => columns of U rotated */
                    const double up = U[k * m + p], uq = U[k * m + q];
                    U[k * m + p] = cs * up - sn * uq;
                    U[k * m + q] = sn * up + cs * uq;
                }
            }
        if (off < 1e-15) break;
    }
    for (int i = 0; i < m; ++i) {
        double nrm = 0;
        for (int k = 0; k < n; ++k) nrm += W[i * n + k] * W[i * n + k];
        nrm = sqrt(nrm);
        s[i] = nrm;
        for (int k = 0; k < n; ++k) V[k * m + i] = nrm > 0 ? W[i * n + k] / nrm : 0.0;
    }
    free(W);
}

/* damp_pseudoinverse(M, lambda) (pik.cpp:5-21): sum_i sigma_i / (lambda^2 + sigma_i^2) v_i u_i^T, n x m row-major */
void iko_damp_pseudoinverse(int m, int n, const double *M, double lambda, double *out) {
    double *U = (double *)malloc(sizeof(double) * m * m), *s = (double *)malloc(sizeof(double) * m);
    double *V = (double *)malloc(sizeof(double) * n * m);
    svd_rows(m, n, M, U, s, V);
    memset(out, 0, sizeof(double) * n * m);
    for (int i = 0; i < m; ++i) {
        const double f = s[i] / (lambda * lambda + s[i] * s[i]);
        for (int r = 0; r < n; ++r)
            for (int c = 0; c < m; ++c) out[r * m + c] += f * V[r * m + i] * U[c * m + i];
    }
    free(U); free(s); free(V);
}

/* M.completeOrthogonalDecomposition().pseudoInverse() * M (pik.cpp:59-61): the orthogonal projector onto the row space of
 * the numerically rank-r part of M (m x n).  Eigen's COD = Householder QR with column pivoting, rank r = number of pivots
 * with |R_kk| > eps * min(m, n) * max_k |R_kk|, then the trailing block is zeroed from the right; pinv(M) M projects onto
 * the span of the first r rows of Q^T M.  Those rows are orthonormalised here (modified Gram-Schmidt, twice) and the
 * projector summed.  Returns r; proj is n x n row-major. */
int iko_rowspace_projector(int m, int n, const double *M, double *proj) {
    double *R = (double *)malloc(sizeof(double) * m * n);
    int *perm = (int *)malloc(sizeof(int) * n);
    memcpy(R, M, sizeof(double) * m * n);
    for (int c = 0; c < n; ++c) perm[c] = c;
    const int steps = m < n ? m : n;
    double maxpiv = 0;
    double *diag = (double *)malloc(sizeof(double) * steps);
    for (int k = 0; k < steps; ++k) {
        /* pivot: the remaining column with the largest norm below row k */
        int best = k;
        double bn = -1;
        for (int c = k; c < n; ++c) {
            double s = 0;
            for (int r = k; r < m; ++r) s += R[r * n + c] * R[r * n + c];
            if (s > bn) { bn = s; best = c; }
        }
        if (best != k) {
            for (int r = 0; r < m; ++r) { double t = R[r * n + k]; R[r * n + k] = R[r * n + best]; R[r * n + best] = t; }
            int t = perm[k]; perm[k] = perm[best]; perm[best] = t;
        }
        /* Householder on column k, rows k.. */
        double nrm = sqrt(bn > 0 ? bn : 0);
        if (nrm == 0) { diag[k] = 0; continue; }
        const double alpha = R[k * n + k] >= 0 ? -nrm : nrm;
        double *v = (double *)malloc(sizeof(double) * m);
        double vn = 0;
        for (int r = k; r < m; ++r) { v[r] = R[r * n + k]; }
        v[k] -= alpha;
        for (int r = k; r < m; ++r) vn += v[r] * v[r];
        if (vn > 0)
            for (int c = k; c < n; ++c) {
                double s = 0;
                for (int r = k; r < m; ++r) s += v[r] * R[r * n + c];
                s = 2 * s / vn;
                for (int r = k; r < m; ++r) R[r * n + c] -= s * v[r];
            }
        free(v);
        diag[k] = fabs(R[k * n + k]);
        if (diag[k] > maxpiv) maxpiv = diag[k];
    }
    int rank = 0;
    const double thr = 2.220446049250313e-16 * (double)steps * maxpiv;
    for (int k = 0; k < steps; ++k)
        if (diag[k] > thr) ++rank;
    /* rows 0..rank-1 of R, columns back in their original order */
    double *W = (double *)malloc(sizeof(double) * (rank > 0 ? rank : 1) * n);
    for (int r = 0; r < rank; ++r)
        for (int c = 0; c < n; ++c) W[r * n + perm[c]] = (c >= r) ? R[r * n + c] : 0.0;
    for (int pass = 0; pass < 2; ++pass)
        for (int r = 0; r < rank; ++r) {
            for (int p = 0; p < r; ++p) {
                double s = 0;
                for (int c = 0; c < n; ++c) s += W[r * n + c] * W[p * n + c];
                for (int c = 0; c < n; ++c) W[r * n + c] -= s * W[p * n + c];
            }
            double nr = 0;
            for (int c = 0; c < n; ++c) nr += W[r * n + c] * W[r * n + c];
            nr = sqrt(nr);
            for (int c = 0; c < n; ++c) W[r * n + c] /= nr;
        }
    memset(proj, 0, sizeof(double) * n * n);
    for (int r = 0; r < rank; ++r)
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) proj[i * n + j] += W[r * n + i] * W[r * n + j];
    free(R); free(perm); free(diag); free(W);
    return rank;
}

/* 1 when every task's priority has a lambda (below IKO_MAX_LEVELS) */
static int pik_levels_ok(const iko_problem *pb) {
    for (int t = 0; t < pb->ntasks; ++t)
        if (pb->priority[t] < 0 || pb->priority[t] >= IKO_MAX_LEVELS) return 0;
    return 1;
}

int iko_pik(const iko_model *m, const iko_problem *pb, const iko_pik_params *prm, const double *q0, const double *targets,
            double *q_out, int *iters, double *resid, double *dq_out) {
    if (!pik_levels_ok(pb)) return -1;
    const int nq = m->nq, nv = m->nv, rows = iko_total_rows(pb), r0 = iko_e_size(pb, 0);
    double *q = (double *)malloc(sizeof(double) * nq), *qn = (double *)malloc(sizeof(double) * nq);
    double *e = (double *)malloc(sizeof(double) * (rows + 1)), *J = (double *)malloc(sizeof(double) * (rows * nv + 1));
    double *P = (double *)malloc(sizeof(double) * nv * nv), *Pj = (double *)malloc(sizeof(double) * nv * nv);
    double *Jbar = (double *)malloc(sizeof(double) * (rows * nv + 1)), *dp = (double *)malloc(sizeof(double) * (rows * nv + 1));
    double *de = (double *)malloc(sizeof(double) * (rows + 1));
    double *dq = (double *)malloc(sizeof(double) * nv), *sdq = (double *)malloc(sizeof(double) * nv);
    memcpy(q, q0, sizeof(double) * nq);                                      /* pik.cpp:34 */
    int success = 0, it = 0;
    double res = 0;
    for (it = 0; it < prm->max_iterations; ++it) {                            /* pik.cpp:39 */
        iko_evaluate(m, pb, q, targets, e, J);                                /* pik.cpp:41 */
        for (int i = 0; i < nv * nv; ++i) P[i] = 0;                           /* pik.cpp:44-45 */
        for (int i = 0; i < nv; ++i) { P[i * nv + i] = 1; dq[i] = 0; }
        int row = 0;
        for (int lvl = 0; lvl <= pb->max_priority_level; ++lvl) {             /* pik.cpp:47 */
            const int mi = iko_e_size(pb, lvl);
            const double *Ji = J + row * nv, *ei = e + row;
            if (mi > 0) {
                for (int r = 0; r < mi; ++r) {                                 /* de_bar = e_i - J_i dq (pik.cpp:49) */
                    double s = 0;
                    for (int c = 0; c < nv; ++c) s += Ji[r * nv + c] * dq[c];
                    de[r] = ei[r] - s;
                }
                for (int r = 0; r < mi; ++r)                                   /* Jbar = J_i P (pik.cpp:51) */
                    for (int c = 0; c < nv; ++c) {
                        double s = 0;
                        for (int k = 0; k < nv; ++k) s += Ji[r * nv + k] * P[k * nv + c];
                        Jbar[r * nv + c] = s;
                    }
                iko_damp_pseudoinverse(mi, nv, Jbar, prm->lambda[lvl], dp);    /* pik.cpp:54-55 */
                for (int c = 0; c < nv; ++c) {
                    double s = 0;
                    for (int r = 0; r < mi; ++r) s += dp[c * mi + r] * de[r];
                    dq[c] -= s;
                }
                iko_rowspace_projector(mi, nv, Jbar, Pj);                      /* pik.cpp:58-61 */
                for (int i = 0; i < nv * nv; ++i) P[i] -= Pj[i];
            }
            row += mi;
        }
        /* dq += P * da with da = 0 (pik.cpp:65, pik.hpp:39) */
        res = 0;                                                              /* visitor.hpp:19 */
        for (int i = 0; i < r0; ++i) res += e[i] * e[i];
        if (res < prm->tolerance) { success = 1; break; }                     /* pik.cpp:67-70 */
        for (int c = 0; c < nv; ++c) sdq[c] = prm->step_length * dq[c];
        iko_integrate(m, q, sdq, qn);                                         /* pik.cpp:73-74 */
        memcpy(q, qn, sizeof(double) * nq);
        iko_clip(m, q);                                                       /* pik.cpp:77 */
    }
    memcpy(q_out, q, sizeof(double) * nq);
    if (iters) *iters = it;
    if (resid) *resid = res;
    if (dq_out) memcpy(dq_out, dq, sizeof(double) * nv);
    free(q); free(qn); free(e); free(J); free(P); free(Pj); free(Jbar); free(dp); free(de); free(dq); free(sdq);
    return success;
}

typedef struct {
    const iko_model *m; const iko_problem *pb; const iko_pik_params *prm;
    int b0, b1;
    const double *q0, *targets;
    double *q_out; unsigned char *success; int *iters; double *resid;
} pik_job;

static void *pik_worker(void *arg) {
    pik_job *j = (pik_job *)arg;
    const int nq = j->m->nq, tsz = iko_target_size(j->pb);
    for (int b = j->b0; b < j->b1; ++b) {
        int it; double r;
        int ok = iko_pik(j->m, j->pb, j->prm, j->q0 + (size_t)b * nq, j->targets + (size_t)b * tsz,
                         j->q_out + (size_t)b * nq, &it, &r, 0);
        j->success[b] = (unsigned char)ok;
        if (j->iters) j->iters[b] = it;
        if (j->resid) j->resid[b] = r;
    }
    return 0;
}

int iko_pik_batch(const iko_model *m, const iko_problem *pb, const iko_pik_params *prm, int B, const double *q0,
                  const double *targets, double *q_out, unsigned char *success, int *iters, double *resid, int nthreads) {
    if (!pik_levels_ok(pb)) return -1;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > B) nthreads = B > 0 ? B : 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * nthreads);
    pik_job *jobs = (pik_job *)malloc(sizeof(pik_job) * nthreads);
    for (int t = 0; t < nthreads; ++t) {
        pik_job jb = {m, pb, prm, (int)((long long)B * t / nthreads), (int)((long long)B * (t + 1) / nthreads),
                      q0, targets, q_out, success, iters, resid};
        jobs[t] = jb;
        if (nthreads == 1) pik_worker(&jobs[t]);
        else pthread_create(&th[t], 0, pik_worker, &jobs[t]);
    }
    if (nthreads > 1)
        for (int t = 0; t < nthreads; ++t) pthread_join(th[t], 0);
    free(th); free(jobs);
    return 0;
}
