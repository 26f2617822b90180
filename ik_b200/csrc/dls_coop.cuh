// Table-driven TEAM-per-problem DLS / PIK iteration: the kernel every problem WITHOUT a compiled specialisation runs on
// (any URDF, any task mix, FrameConstraints, CentreOfMassTask, ik::pik) -- the replacement of the thread-per-problem
// local-memory design of dls_generic.cuh (0.9 % of the FP64 roofline, 1 200x wasted DRAM traffic; VERDICT r1 item 5).
//
// A TEAM of 8 / 16 / 32 lanes (by size class) shares ONE problem.  Nothing lives in local memory: the iterate, the joint
// placements, the weighted task Jacobian and the exchange buffers sit in a per-team block of shared memory, the Gram
// matrix and its factorisation in the lanes' REGISTERS (row r of J J^T + damping^2 I belongs to lane r mod TEAM), and
// the pivot column travels by warp shuffle (north_star: "in-register Cholesky built on warp shuffles") or, as a
// compile-time alternative, through a double-buffered shared-memory column (SHFL = false; both measured, DESIGN.md).
// Every phase of ik::dls (reference dls.cpp:14-74) is split by DATA over the lanes (SPMD, __syncwarp between phases):
//
//   phase 0  lane <-> joint: sin / cos of the revolute coordinates of the joints some task needs (a continuous joint's
//            q already holds them)
//   phase 1  lane <-> (root-to-leaf path, row i): world placements by ROWS -- row i of R_world(j) and component i of
//            p_world(j) depend only on row i of the parent's rotation, so a lane walks its path without communication,
//            applying placement and joint motion on the fly                                     (data.cpp:28-29)
//   (1b)     CentreOfMassTask only: subtree masses / first moments, leaves to root              (data.cpp:31-34)
//   phase 2  lane <-> task: frame placements, SE3-log error (frame.hpp:37-62), Jlog6 blocks folded with the frame
//            rotation into one (X_r, Y_r) pair of 3-vectors per task ROW: J[r][c] = X_r . d_c + Y_r . w_c with
//            (d_c, w_c) the world twist of column c about the task frame's origin            (frame.hpp:152-182)
//   phase 3  lane <-> (task, supporting column): the weighted Jacobian entries of that column    (data.cpp:49-50)
//   phase 4  lane <-> row: Gram rows J J^T + damping^2 I from the column-major J in shared memory  (dls.cpp:39-41)
//   phase 5  Gauss-Jordan elimination by rows, no pivoting (the matrix is SPD thanks to the damping): per pivot k the
//            column-k entries are broadcast, every lane eliminates its own rows, the right-hand side e rides along;
//            what is left is diagonal, so y needs no substitution pass                        (dls.cpp:53, ldlt().solve)
//   phase 6  lane <-> column: dq = -J^T y (dls.cpp:52); FrameConstraints: dq <- (I - Jc^+ Jc) dq  (dls.cpp:26-34,44-52)
//   phase 7  stop test (visitor.hpp:19), lane <-> joint: integrate + clamp                        (dls.cpp:61-71)
//
// ik::pik (pik.cpp:31-96) replaces phases 4-6 by the priority recursion (one damped solve and one rank-revealing
// row-space basis per level), built from the same row / column primitives.
//
// The body is __host__ __device__ and takes lane exchange (sync, shfl) from a context object, so tests/cpu_harness runs
// the very same source with TEAM host threads, a std::barrier and an exchange array, and checks it against the oracle
// on the GPU-less build box.
#pragma once
#include "../../include/ikb200.h"
#include "dev_problem.hpp"
#include "joint_types.hpp"
#include "se3_math.cuh"

namespace ikb {

template <int NJ_, int NV_, int M_, int TEAM_> struct CoopCfg {
    static constexpr int NJ = NJ_, NV = NV_, M = M_, TEAM = TEAM_;
    static constexpr int RPL = (M + TEAM - 1) / TEAM;           // Gram rows per lane
    static constexpr int LD = (M % 4 == 2) ? M : M + 2;         // column stride of J: even (16-byte rows) and = 2 mod 4 (banks)
    static constexpr int NQ = NV + 4;
    static constexpr int TSZ = 4 * M;                           // target scalars: at most 12 per 3 rows
    static constexpr int NBLK = (M + 5) / 6;                    // row blocks of 6 (col_rows sparsity test)
    static constexpr int LDX = LD > kMaxConstraintRows ? LD : kMaxConstraintRows + 2;  // column stride of Jb / Jc
    static_assert(M % 2 == 0 && RPL * TEAM >= M, "row classes are even");
};

// Size classes (shared with the thread-per-problem fallback, ikb_capi.cu kClasses): capacities and team width.
template <int CLS> struct CoopClass;
template <> struct CoopClass<0> { using Cfg = CoopCfg<10, 8, 6, 8>; };      // serial arms, one or two frame tasks
template <> struct CoopClass<1> { using Cfg = CoopCfg<20, 24, 12, 16>; };   // Cassie-sized: 12 rows, half a warp per problem
template <> struct CoopClass<2> { using Cfg = CoopCfg<32, 36, 30, 32>; };   // humanoid-sized: 30 rows, a warp per problem
// (coop kernel only; ikb_solve.cu picks it for class-2 problems on a small tree) Cassie-sized TREE with up to 30 rows -- the
// demo's task set with its posture level, ik::pik on it: the scratch shrinks from 17.6 / 38.8 KB to 13.1 / 27.1 KB per team
template <> struct CoopClass<3> { using Cfg = CoopCfg<20, 24, 30, 32>; };

// Per-team block of shared memory.  EXTRA = 0: plain ik::dls; 1: + the subtree mass / moment arrays of a
// CentreOfMassTask; 2: + the buffers only ik::pik and FrameConstraints need (projected Jacobian, row-space bases) -- each
// level costs residency, so a problem gets the smallest scratch that serves it.
template <typename T, class Cfg, int EXTRA> struct alignas(16) CoopScratch {
    T Jt[Cfg::NV][Cfg::LD];   // weighted stacked task Jacobian, column-major; structural zeros are written once per kernel
    T sc[Cfg::NJ][2];         // (sin, cos) of every needed revolute or continuous joint's coordinate
    T oM[Cfg::NJ][12];        // oMi: R row-major (9) + p (3)
    T XY[Cfg::M][6];          // per task row: X (3), Y (3)
    T tpf[Cfg::M][3];         // per task: world origin of the task frame
    T q[Cfg::NQ];
    T tg[Cfg::TSZ];
    T e[Cfg::M + 2], y[Cfg::M + 2];
    T dq[Cfg::NV];
    T piv[2][Cfg::M + 2];     // SHFL = false: pivot column (+ right-hand side entry), double-buffered
    T ms[EXTRA >= 1 ? Cfg::NJ : 1], mc[EXTRA >= 1 ? Cfg::NJ : 1][3], ctot[4];   // CentreOfMassTask: subtree mass, first moment, whole-body first moment
    T W[EXTRA >= 2 ? Cfg::M + kMaxConstraintRows : 1][Cfg::NV];  // ik::pik / FrameConstraint: orthonormal row-space bases (row-major)
    T Jb[EXTRA >= 2 ? Cfg::NV : 1][Cfg::LDX];   // ik::pik: projected level Jacobian, column-major; FrameConstraint: Jc (rows <= 12)
};

// World twist of velocity coordinate cc of joint j (data.cpp:30: oMi.act(S_i)) as (axis direction `ax`, origin `p`):
// angular coordinates (revolute, continuous, free-flyer 3-5) give (v, w) = (p x ax, ax), linear ones (prismatic, free-flyer
// 0-2) (ax, 0).
template <typename T> IKB_HD bool coop_world_axis(const DevProblem<T> &P, int j, int cc, const T *O, T *ax) {
    const int jt = P.jtype[j];
    if (jt == IKB_J_FREEFLYER) {
        const int k = cc % 3;
        ax[0] = O[k]; ax[1] = O[3 + k]; ax[2] = O[6 + k];
        return cc >= 3;
    }
    const int k = axis_index(jt);
    if (k >= 0) {
        ax[0] = O[k]; ax[1] = O[3 + k]; ax[2] = O[6 + k];
    } else {
        rot_vec(O, P.axis[j], ax);
    }
    return is_revolute_like(jt);
}

// World placement of used frame f (common.hpp:47-51: data.oMf[id]): oMi[parent] * placement, without the product when the
// placement is the identity.
template <typename T, class SCR> IKB_HD void coop_frame_placement(const DevProblem<T> &P, const SCR &S, int f, T *R, T *p) {
    const int fj = P.f_parent[f];
    const T *O = S.oM[fj];
    if (P.coop.f_ident[f]) {
        for (int i = 0; i < 9; ++i) R[i] = O[i];
        p[0] = O[9]; p[1] = O[10]; p[2] = O[11];
    } else {
        se3_mul(O, O + 9, P.f_placement[f], P.f_placement[f] + 9, R, p);
    }
}

// ---- phases 0-3: evaluate_problem_data (data.cpp:25-58) -> S.e (weighted), S.Jt (weighted, column-major) ----
template <typename T, class Cfg, int EXTRA, class Ctx>
IKB_HD void coop_evaluate(const Ctx &cx, const DevProblem<T> &P, CoopScratch<T, Cfg, EXTRA> &S) {
    constexpr int TEAM = Cfg::TEAM;
    const CoopTables &C = P.coop;
    const int lane = cx.lane;
    // phase 0: lane <-> joint, sin / cos of the revolute coordinates; a continuous joint's q is (cos, sin) as given (Pinocchio's
    // JointModelRevoluteUnbounded::calc neither evaluates nor renormalises it)
    for (int i = lane; i < C.n_fkj; i += TEAM) {
        const int j = C.fkj[i], t = P.jtype[j];
        if (is_revolute(t)) sincos_(S.q[P.idx_q[j]], &S.sc[j][0], &S.sc[j][1]);
        else if (is_continuous(t)) { S.sc[j][0] = S.q[P.idx_q[j] + 1]; S.sc[j][1] = S.q[P.idx_q[j]]; }
    }
    cx.sync();
    // phase 1: lane <-> (path, row i).  oMi = oMi[parent] * placement * M_j(q) by rows: with r = row i of the parent's
    // rotation, a = r * placement.R is row i of (parent * placement) and the joint motion mixes two of its entries
    // (aligned revolutes), multiplies it by the free-flyer's rotation, or leaves it alone (prismatic).  A continuous joint
    // moves as the revolute joint with its axis, from the (sin, cos) of phase 0.
    for (int w = lane; w < 3 * C.npaths; w += TEAM) {
        const int p = w / 3, i = w - 3 * p;
        T r0 = i == 0 ? T(1) : T(0), r1 = i == 1 ? T(1) : T(0), r2 = i == 2 ? T(1) : T(0), pp = T(0);
        const int len = C.path_len[p];
        for (int k = 0; k < len; ++k) {
            const int j = C.path_joint[p][k], t = as_revolute(P.jtype[j]);
            const T *PR = P.placement[j];
            const T a0 = r0 * PR[0] + r1 * PR[3] + r2 * PR[6];
            const T a1 = r0 * PR[1] + r1 * PR[4] + r2 * PR[7];
            const T a2 = r0 * PR[2] + r1 * PR[5] + r2 * PR[8];
            pp = pp + (r0 * PR[9] + r1 * PR[10] + r2 * PR[11]);
            if (t == IKB_J_RZ) {
                const T s = S.sc[j][0], c = S.sc[j][1];
                r0 = a0 * c + a1 * s; r1 = a1 * c - a0 * s; r2 = a2;
            } else if (t == IKB_J_RX) {
                const T s = S.sc[j][0], c = S.sc[j][1];
                r0 = a0; r1 = a1 * c + a2 * s; r2 = a2 * c - a1 * s;
            } else if (t == IKB_J_RY) {
                const T s = S.sc[j][0], c = S.sc[j][1];
                r0 = a0 * c - a2 * s; r1 = a1; r2 = a0 * s + a2 * c;
            } else if (t == IKB_J_FREEFLYER) {
                const T *qj = S.q + P.idx_q[j];
                T Rq[9];
                quat_to_rot(qj[3], qj[4], qj[5], qj[6], Rq);
                pp = pp + (a0 * qj[0] + a1 * qj[1] + a2 * qj[2]);
                r0 = a0 * Rq[0] + a1 * Rq[3] + a2 * Rq[6];
                r1 = a0 * Rq[1] + a1 * Rq[4] + a2 * Rq[7];
                r2 = a0 * Rq[2] + a1 * Rq[5] + a2 * Rq[8];
            } else if (t == IKB_J_REV_UNALIGNED) {
                const T s = S.sc[j][0], c = S.sc[j][1], v = 1 - c;
                const T *ax = P.axis[j];
                const T R00 = ax[0] * ax[0] * v + c, R01 = ax[0] * ax[1] * v - ax[2] * s, R02 = ax[0] * ax[2] * v + ax[1] * s;
                const T R10 = ax[0] * ax[1] * v + ax[2] * s, R11 = ax[1] * ax[1] * v + c, R12 = ax[1] * ax[2] * v - ax[0] * s;
                const T R20 = ax[0] * ax[2] * v - ax[1] * s, R21 = ax[1] * ax[2] * v + ax[0] * s, R22 = ax[2] * ax[2] * v + c;
                r0 = a0 * R00 + a1 * R10 + a2 * R20;
                r1 = a0 * R01 + a1 * R11 + a2 * R21;
                r2 = a0 * R02 + a1 * R12 + a2 * R22;
            } else {   // prismatic: the rotation is the placement's, the origin moves along the joint axis
                const T qd = S.q[P.idx_q[j]];
                const T d = t == IKB_J_PX ? a0 : (t == IKB_J_PY ? a1 : (t == IKB_J_PZ ? a2 : a0 * P.axis[j][0] + a1 * P.axis[j][1] + a2 * P.axis[j][2]));
                pp = pp + d * qd;
                r0 = a0; r1 = a1; r2 = a2;
            }
            T *O = S.oM[j];
            O[3 * i] = r0; O[3 * i + 1] = r1; O[3 * i + 2] = r2; O[9 + i] = pp;
        }
    }
    cx.sync();
    // phase 1b: centre of mass (centre_of_mass.hpp:24-38; pinocchio::jacobianCenterOfMass)
    if constexpr (EXTRA >= 1) if (C.has_com) {
        for (int j = 1 + lane; j < P.njoints; j += TEAM) {
            T cw[3];
            rot_vec(S.oM[j], P.com[j], cw);
            S.ms[j] = P.mass[j];
            for (int i = 0; i < 3; ++i) S.mc[j][i] = P.mass[j] * (cw[i] + S.oM[j][9 + i]);
        }
        cx.sync();
        if (lane < 4) {  // joints are stored parents first: one backward sweep; lanes 0-2 the moment components, lane 3 the mass
            T tot = T(0);
            for (int j = P.njoints - 1; j >= 1; --j) {
                const int par = P.parent[j];
                if (lane < 3) {
                    if (par > 0) S.mc[par][lane] += S.mc[j][lane];
                    else tot += S.mc[j][lane];
                } else if (par > 0) {
                    S.ms[par] += S.ms[j];
                }
            }
            if (lane < 3) S.ctot[lane] = tot;
        }
        cx.sync();
    }
    // phase 2
    const int nq = P.nq, nv = P.nv;
    for (int t = lane; t < P.ntasks; t += TEAM) {
        const int row = P.t_row[t], kind = P.t_kind[t], toff = P.t_toff[t];
        const T *wgt = P.weight + row;
        if (kind == IKB_TASK_POSTURE) {  // posture.hpp:50-67: e = (q.bottomRows(nj) - target) o mask; J = [0 I] (constant, set once)
            const int nj = P.t_type[t];
            for (int i = 0; i < nj; ++i) S.e[row + i] = (S.q[nq - nj + i] - S.tg[toff + i]) * P.mask[P.t_moff[t] + i] * wgt[i];
            continue;
        }
        const int r = P.t_ref[t];
        const bool ref_universe = C.f_ident[r] == 2;
        T Rr[9], pr[3];
        coop_frame_placement(P, S, r, Rr, pr);
        if (kind == IKB_TASK_COM) {
            const T inv_m = T(1) / P.total_mass;
            T d[3], lc[3];
            for (int i = 0; i < 3; ++i) d[i] = S.ctot[i] * inv_m - pr[i];
            rotT_vec(Rr, d, lc);
            for (int i = 0; i < 3; ++i) {
                S.e[row + i] = (lc[i] - S.tg[toff + i]) * wgt[i];
                T *xy = S.XY[row + i];   // J row i = w_i * (column i of Rr) . vel
                xy[0] = wgt[i] * Rr[i]; xy[1] = wgt[i] * Rr[3 + i]; xy[2] = wgt[i] * Rr[6 + i];
                xy[3] = xy[4] = xy[5] = T(0);
            }
            continue;
        }
        const int f = P.t_frame[t];
        T Rf[9], pf[3];
        coop_frame_placement(P, S, f, Rf, pf);
        S.tpf[t][0] = pf[0]; S.tpf[t][1] = pf[1]; S.tpf[t][2] = pf[2];
        if (kind == IKB_TASK_FRAME) {
            T Rt[9], pt[3], Rtg[9], ptg[3];
            for (int i = 0; i < 9; ++i) Rtg[i] = S.tg[toff + i];
            for (int i = 0; i < 3; ++i) ptg[i] = S.tg[toff + 9 + i];
            if (ref_universe) {                  // oMt = oMr * target (frame.hpp:48) with oMr = identity
                for (int i = 0; i < 9; ++i) Rt[i] = Rtg[i];
                pt[0] = ptg[0]; pt[1] = ptg[1]; pt[2] = ptg[2];
            } else {
                se3_mul(Rr, pr, Rtg, ptg, Rt, pt);
            }
            T Re[9], pe[3], w[3], th, sth, cth, lin[3];
            se3_actinv(Rf, pf, Rt, pt, Re, pe);  // fMt (frame.hpp:50)
            log3(Re, w, th, sth, cth);
            const LogCoeffs<T> lc = log_coeffs(th, sth, cth);
            log6_from(w, lc, pe, lin);
            // tMf = fMt^-1: rotation Re^T (log3 = -w, same angle), translation Rt^T (pf - pt)   (frame.hpp:160-166)
            const T nw[3] = {-w[0], -w[1], -w[2]}, nd[3] = {pf[0] - pt[0], pf[1] - pt[1], pf[2] - pt[2]};
            T p2[3], A[9], Bm[9];
            rotT_vec(Rt, nd, p2);
            jlog6_blocks(nw, th, lc, p2, A, Bm);
            const int ktype = P.t_type[t];
            // rows of -Jlog6(tMf) * Jf_LOCAL: top_i = -(A Rf^T)_i . d - (B Rf^T)_i . w, bottom_i = -(A Rf^T)_i . w
            for (int i = 0; i < 3; ++i) {
                T ma[3], mb[3];
                for (int k = 0; k < 3; ++k) {
                    ma[k] = A[3 * i] * Rf[3 * k] + A[3 * i + 1] * Rf[3 * k + 1] + A[3 * i + 2] * Rf[3 * k + 2];
                    mb[k] = Bm[3 * i] * Rf[3 * k] + Bm[3 * i + 1] * Rf[3 * k + 1] + Bm[3 * i + 2] * Rf[3 * k + 2];
                }
                if (ktype != IKB_ORIENTATION) {
                    const T wi = wgt[i];
                    S.e[row + i] = lin[i] * wi;
                    T *xy = S.XY[row + i];
                    for (int k = 0; k < 3; ++k) { xy[k] = -wi * ma[k]; xy[3 + k] = -wi * mb[k]; }
                }
                if (ktype != IKB_POSITION) {
                    const int ro = row + i + (ktype == IKB_FULL ? 3 : 0);
                    const T wi = P.weight[ro];
                    S.e[ro] = w[i] * wi;
                    T *xy = S.XY[ro];
                    for (int k = 0; k < 3; ++k) { xy[k] = T(0); xy[3 + k] = -wi * ma[k]; }
                }
            }
        } else {  // IKB_TASK_ALIGN_AXIS (frame.hpp:246-299): e = 1 - r . t^, J = -(r x t^)^T R_rMf Jf_LOCAL.bottomRows(3)
            T Rm[9], pm[3];
            se3_actinv(Rr, pr, Rf, pf, Rm, pm);
            const int ax = P.t_type[t];
            const T rv[3] = {Rm[ax], Rm[3 + ax], Rm[6 + ax]};
            T tn[3] = {S.tg[toff], S.tg[toff + 1], S.tg[toff + 2]};
            const T n = sqrt_(dot3(tn, tn));
            tn[0] /= n; tn[1] /= n; tn[2] /= n;
            S.e[row] = (T(1) - dot3(rv, tn)) * wgt[0];
            T rxt[3], r3[3], g3[3];
            cross3(rv, tn, rxt);
            rotT_vec(Rm, rxt, r3);
            rot_vec(Rf, r3, g3);   // -(r3 . Rf^T w) = -(Rf r3) . w
            T *xy = S.XY[row];
            for (int k = 0; k < 3; ++k) { xy[k] = T(0); xy[3 + k] = -wgt[0] * g3[k]; }
        }
    }
    cx.sync();
    // phase 3
    for (int w = lane; w < C.npairs; w += TEAM) {
        const int t = C.pair_task[w], j = C.pair_joint[w], cc = C.pair_cc[w];
        const T *O = S.oM[j];
        T ax[3];
        const bool angular = coop_world_axis(P, j, cc, O, ax);
        const int row = P.t_row[t], dim = P.t_dim[t];
        T *col = S.Jt[P.idx_v[j] + cc] + row;
        if (P.t_kind[t] == IKB_TASK_COM) {
            // velocity this coordinate gives the centre of mass of its subtree, weighted by the subtree's share of the mass
            T vel[3] = {T(0), T(0), T(0)};
            if constexpr (EXTRA >= 1) if (S.ms[j] > T(0)) {
                const T share = S.ms[j] / P.total_mass, ims = T(1) / S.ms[j];
                if (angular) {
                    const T dc[3] = {S.mc[j][0] * ims - O[9], S.mc[j][1] * ims - O[10], S.mc[j][2] * ims - O[11]};
                    cross3(ax, dc, vel);   // p x w + w x cs = w x (cs - p)
                } else {
                    vel[0] = ax[0]; vel[1] = ax[1]; vel[2] = ax[2];
                }
                vel[0] *= share; vel[1] *= share; vel[2] *= share;
            }
            for (int i = 0; i < dim; ++i) col[i] = dot3(S.XY[row + i], vel);
        } else {
            T d[3], ww[3];
            if (angular) {
                const T dp[3] = {O[9] - S.tpf[t][0], O[10] - S.tpf[t][1], O[11] - S.tpf[t][2]};
                cross3(dp, ax, d);
                ww[0] = ax[0]; ww[1] = ax[1]; ww[2] = ax[2];
            } else {
                d[0] = ax[0]; d[1] = ax[1]; d[2] = ax[2];
                ww[0] = ww[1] = ww[2] = T(0);
            }
            for (int i = 0; i < dim; ++i) {
                const T *xy = S.XY[row + i];
                col[i] = dot3(xy, d) + dot3(xy + 3, ww);
            }
        }
    }
    (void)nv;
    cx.sync();
}

template <typename T> struct alignas(2 * sizeof(T)) Pair { T x, y; };   // one 128-bit (64-bit for float) shared-memory access

// Broadcast of one scalar per row: either by shuffle from the owner lane's register or through shared memory.
// Gram rows + Gauss-Jordan solve of (Jm Jm^T + lambda2 I) y = rhs for rows [0, M) of the column-major matrix Jm (rows
// beyond the problem's are structurally zero: they factor to lambda2 and give y = 0).  Lane owns rows lane + rr * TEAM.
// On return y_out[rr] holds the solution entries of the lane's rows.
template <typename T, class Cfg, bool SHFL, int LDM, bool SKIP, class Ctx>
IKB_HD void coop_gram_solve(const Ctx &cx, const T (*Jm)[LDM], const uint64_t *col_rows, int nv, const T *rhs_in, int nrhs, T lambda2,
                            T (*piv)[Cfg::M + 2], T *y_out) {
    constexpr int TEAM = Cfg::TEAM, M = Cfg::M, RPL = Cfg::RPL;
    const int lane = cx.lane;
    T g[RPL][M];
    T rhs[RPL], yinv[RPL];
#pragma unroll
    for (int rr = 0; rr < RPL; ++rr) {
#pragma unroll
        for (int b = 0; b < M; ++b) g[rr][b] = T(0);
        const int r = lane + rr * TEAM;
        rhs[rr] = r < nrhs ? rhs_in[r] : T(0);
        yinv[rr] = T(0);
    }
    // rows >= nrhs are structurally zero.  SKIP (the levels of ik::pik, 10 + 16 rows in a 30-row size class): their Gram
    // blocks and their pivots (identity rows, multipliers exactly 0) are skipped.  Not for ik::dls, whose problems fill their
    // size class: the per-pivot test costs the straight-line pivot loop its schedule (measured: Cassie 3.06 -> 3.94 ms).
    const uint64_t live = (!SKIP || nrhs >= 60) ? ~0ULL : (1ULL << (6 * ((nrhs + 5) / 6))) - 1ULL;
    // ---- Gram (dls.cpp:39): columns in ascending order, only row blocks the column can touch ----
    for (int c = 0; c < nv; ++c) {
        const T *col = Jm[c];
        const uint64_t mask = (col_rows ? col_rows[c] : ~0ULL) & live;
        T a[RPL];
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = lane + rr * TEAM;
            a[rr] = r < M ? col[r] : T(0);
        }
#pragma unroll
        for (int blk = 0; blk < Cfg::NBLK; ++blk) {
            if ((mask >> (6 * blk)) & 63ULL) {
#pragma unroll
                for (int b = 6 * blk; b < (6 * blk + 6 < M ? 6 * blk + 6 : M); b += 2) {   // M, LDM even: 16-byte pairs
                    const Pair<T> v = *reinterpret_cast<const Pair<T> *>(col + b);
#pragma unroll
                    for (int rr = 0; rr < RPL; ++rr) {
                        g[rr][b] += a[rr] * v.x;
                        g[rr][b + 1] += a[rr] * v.y;
                    }
                }
            }
        }
    }
#pragma unroll
    for (int rr = 0; rr < RPL; ++rr) {
        const int r = lane + rr * TEAM;
#pragma unroll
        for (int b = 0; b < M; ++b) g[rr][b] += (b == r) ? (r < nrhs ? lambda2 : T(1)) : T(0);   // dls.cpp:41 (identity on unused rows)
    }
    // ---- Gauss-Jordan by rows ----
#pragma unroll
    for (int k = 0; k < M; ++k) {
        if (SKIP && k >= nrhs) break;   // (uniform: nrhs is a property of the problem)
        const int ko = k % TEAM, kr = k / TEAM;
        T d, ek;
        T *pv = piv[k & 1];
        if constexpr (SHFL) {
            d = cx.shfl(g[kr][k], ko);
            ek = cx.shfl(rhs[kr], ko);
        } else {
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr) {
                const int r = lane + rr * TEAM;
                if (r < M) pv[r] = g[rr][k];
            }
            if (lane == ko) pv[M] = rhs[kr];
            cx.sync();
            d = pv[k];
            ek = pv[M];
        }
        const T inv = rcp_(d);
        T f[RPL];
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = lane + rr * TEAM;
            f[rr] = (r == k) ? T(0) : g[rr][k] * inv;
        }
        if constexpr (SHFL) {
#pragma unroll
            for (int b = k + 1; b < M; ++b) {
                const T pb = cx.shfl(g[b / TEAM][k], b % TEAM);   // G[k][b] = G[b][k]: the trailing block stays symmetric
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr) g[rr][b] -= f[rr] * pb;
            }
        } else {
            const int first_pair = (k + 2) & ~1;   // first even index > k (k is a constant once the pivot loop is unrolled)
            if ((k + 1) & 1) {
                const T pb = pv[k + 1];
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr) g[rr][k + 1] -= f[rr] * pb;
            }
#pragma unroll
            for (int b = first_pair; b < M; b += 2) {
                const Pair<T> pb = *reinterpret_cast<const Pair<T> *>(pv + b);
#pragma unroll
                for (int rr = 0; rr < RPL; ++rr) {
                    g[rr][b] -= f[rr] * pb.x;
                    g[rr][b + 1] -= f[rr] * pb.y;
                }
            }
        }
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) rhs[rr] -= f[rr] * ek;
        if (lane == ko) yinv[kr] = inv;
    }
#pragma unroll
    for (int rr = 0; rr < RPL; ++rr) y_out[rr] = rhs[rr] * yinv[rr];
}

// Trip count of a loop whose body holds warp collectives (shfl, sync) and whose natural count `n` is per-problem data: the
// largest `n` of the warp.  Teams of 8 or 16 lanes share a warp, and the full-mask collectives pair up the instructions of
// all its lanes: a team that issued fewer of them than its neighbour (a level of lower rank, a team without a problem on its
// placeholder state) would leave the neighbour waiting for good.  Trips beyond a team's own `n` do no work.
template <class Ctx> IKB_HD int coop_warp_rounds(const Ctx &cx, int n) { return cx.warp_max(n); }

// Orthonormal basis (rows of Wout, returned count = rank) of the row space of the numerically rank-r part of the mi x nv
// matrix A (column-major with stride LD, destroyed): what A.completeOrthogonalDecomposition().pseudoInverse() * A projects
// onto (pik.cpp:59-61, dls.cpp:44-49).  Householder QR with column pivoting, lane <-> column; rank from Eigen's threshold
// eps * min(m, n) * max pivot; the first r rows of R (columns back in place) orthonormalised by Gram-Schmidt with re-orthogonalisation.
template <typename T, class Cfg, class Ctx>
IKB_HD int coop_rowspace_basis(const Ctx &cx, T (*A)[Cfg::LDX], int mi, int nv, T (*Wout)[Cfg::NV], T *diag /* >= mi */) {
    constexpr int TEAM = Cfg::TEAM;
    const int lane = cx.lane;
    // column c of the permuted matrix lives in storage column perm[c]; every lane keeps the whole permutation (tiny)
    unsigned char perm[Cfg::NV];
    for (int c = 0; c < nv; ++c) perm[c] = (unsigned char)c;
    const int steps = mi < nv ? mi : nv;
    T maxpiv = T(0);
    for (int k = 0; k < steps; ++k) {
        // pivot: the column (among k..nv-1) with the largest remaining norm; ties -> lowest index (as a serial scan with >)
        T bn = T(-1);
        int best = k;
        for (int c = k + lane; c < nv; c += TEAM) {
            const T *col = A[perm[c]];
            T s = T(0);
            for (int r = k; r < mi; ++r) s += col[r] * col[r];
            if (s > bn) { bn = s; best = c; }
        }
        for (int off = TEAM / 2; off >= 1; off >>= 1) {
            const T obn = cx.shfl(bn, lane ^ off);
            const int obest = (int)cx.shfl((T)best, lane ^ off);
            if (obn > bn || (obn == bn && obest < best)) { bn = obn; best = obest; }
        }
        if (best != k) { const unsigned char t = perm[k]; perm[k] = perm[best]; perm[best] = t; }
        // Every branch below is data-dependent; the warp collectives are not (see coop_warp_rounds): 3 syncs per column.
        const T nrm = sqrt_(max_(bn, T(0)));
        const bool live = nrm > T(0);   // false for a zero (or NaN) remainder: pivot 0
        T *ck = A[perm[k]];
        const T akk = ck[k];
        const T alpha = akk >= T(0) ? -nrm : nrm;
        // v = column k below the diagonal, v[k] -= alpha; |v|^2 = 2 nrm (nrm + |akk|) (exactly what the serial sum gives up to rounding)
        T vn = T(0);
        if (live)
            for (int r = k; r < mi; ++r) {
                const T v = ck[r] - (r == k ? alpha : T(0));
                vn += v * v;
            }
        cx.sync();   // everybody has read column k before its owner overwrites it
        const bool reflect = live && vn > T(0);
        if (reflect) {
            const T two_over = T(2) / vn;
            for (int c = k + 1 + lane; c < nv; c += TEAM) {
                T *col = A[perm[c]];
                T s = T(0);
                for (int r = k; r < mi; ++r) s += (ck[r] - (r == k ? alpha : T(0))) * col[r];
                s *= two_over;
                for (int r = k; r < mi; ++r) col[r] -= s * (ck[r] - (r == k ? alpha : T(0)));
            }
        }
        cx.sync();
        if (lane == 0) {
            if (reflect) {   // column k itself becomes (alpha, 0, ..., 0)
                ck[k] = alpha;
                for (int r = k + 1; r < mi; ++r) ck[r] = T(0);
            }
            diag[k] = live ? abs_(alpha) : T(0);
        }
        if (live) maxpiv = max_(maxpiv, abs_(alpha));
        cx.sync();
    }
    const T eps = sizeof(T) == 8 ? T(2.220446049250313e-16) : T(1.1920929e-7);
    const T thr = eps * T(steps) * maxpiv;
    int rank = 0;
    for (int k = 0; k < steps; ++k) rank += diag[k] > thr ? 1 : 0;
    // W[r][perm[c]] = R[r][c] (c >= r), lane <-> column
    for (int c = lane; c < nv; c += TEAM)
        for (int r = 0; r < rank; ++r) Wout[r][perm[c]] = c >= r ? A[perm[c]][r] : T(0);
    cx.sync();
    // Classical Gram-Schmidt with re-orthogonalisation ("twice is enough"), row by row against the finished rows.  The r
    // dot products of a row are taken by r lanes at once (lane <-> finished row, serial over the columns, no reduction
    // across lanes) and the update by lane <-> column; one butterfly per row (its norm) instead of one per PAIR of rows and
    // pass -- the modified Gram-Schmidt that stood here spent a third of an ik::pik iteration in shuffles
    // (profiles/r2_s3_pik_lines.txt).  `diag` is free once the rank is known and carries the coefficients.
    const int rounds = coop_warp_rounds(cx, rank);
    for (int r = 0; r < rounds; ++r) {
        const bool live = r < rank;
        for (int pass = 0; pass < 2 && r > 0; ++pass) {
            if (live)
                for (int p2 = lane; p2 < r; p2 += TEAM) {
                    T s0 = T(0), s1 = T(0);
                    int c = 0;
                    for (; c + 1 < nv; c += 2) {
                        s0 += Wout[r][c] * Wout[p2][c];
                        s1 += Wout[r][c + 1] * Wout[p2][c + 1];
                    }
                    if (c < nv) s0 += Wout[r][c] * Wout[p2][c];
                    diag[p2] = s0 + s1;
                }
            cx.sync();
            if (live)
                for (int c = lane; c < nv; c += TEAM) {
                    T w = Wout[r][c];
                    for (int p2 = 0; p2 < r; ++p2) w -= diag[p2] * Wout[p2][c];
                    Wout[r][c] = w;
                }
            cx.sync();
        }
        T nr = T(0);
        if (live)
            for (int c = lane; c < nv; c += TEAM) nr += Wout[r][c] * Wout[r][c];
        for (int off = TEAM / 2; off >= 1; off >>= 1) nr += cx.shfl(nr, lane ^ off);
        if (live) {
            const T inr = T(1) / sqrt_(nr);
            for (int c = lane; c < nv; c += TEAM) Wout[r][c] *= inr;
        }
        cx.sync();
    }
    cx.sync();
    return rank;
}

// Stacked FrameConstraint Jacobian (frame.hpp:398-440) into Jc (column-major): frame Jacobian minus the reference frame's
// moved by rMf^-1, both LOCAL, rows by KinematicType.  lane <-> (constraint, column).
template <typename T, class Cfg, int EXTRA, class Ctx>
IKB_HD void coop_constraint_jacobian(const Ctx &cx, const DevProblem<T> &P, CoopScratch<T, Cfg, EXTRA> &S) {
    constexpr int TEAM = Cfg::TEAM;
    const int lane = cx.lane, nv = P.nv;
    for (int c = lane; c < nv; c += TEAM)
        for (int r = 0; r < P.crows; ++r) S.Jb[c][r] = T(0);
    cx.sync();
    int crow = 0;
    for (int k = 0; k < P.nconstraints; ++k) {
        const int f = P.c_frame[k], r = P.c_ref[k], fj = P.f_parent[f], rj = P.f_parent[r];
        const int full = P.c_type[k] == IKB_FULL, r0 = P.c_type[k] == IKB_ORIENTATION ? 3 : 0, dim = full ? 6 : 3;
        T Rf[9], pf[3], Rr[9], pr[3], Rm[9], pm[3];
        coop_frame_placement(P, S, f, Rf, pf);
        coop_frame_placement(P, S, r, Rr, pr);
        se3_actinv(Rr, pr, Rf, pf, Rm, pm);  // rMf (frame.hpp:407)
        // the two chains are walked by every lane; a lane handles the velocity coordinates it owns (col % TEAM == lane)
        for (int pass = 0; pass < 2; ++pass) {
            for (int j = pass == 0 ? fj : rj; j > 0; j = P.parent[j]) {
                const int ncol = P.jtype[j] == IKB_J_FREEFLYER ? 6 : 1;
                for (int cc = 0; cc < ncol; ++cc) {
                    const int col = P.idx_v[j] + cc;
                    if (col % TEAM != lane) continue;
                    T ax[3], v[3], ww[3], pxw[3], d[3], out[6];
                    const bool angular = coop_world_axis(P, j, cc, S.oM[j], ax);
                    if (angular) { cross3(S.oM[j] + 9, ax, v); ww[0] = ax[0]; ww[1] = ax[1]; ww[2] = ax[2]; }
                    else { v[0] = ax[0]; v[1] = ax[1]; v[2] = ax[2]; ww[0] = ww[1] = ww[2] = T(0); }
                    if (pass == 0) {  // + frame Jacobian, LOCAL (frame.hpp:410-411)
                        cross3(pf, ww, pxw);
                        d[0] = v[0] - pxw[0]; d[1] = v[1] - pxw[1]; d[2] = v[2] - pxw[2];
                        rotT_vec(Rf, d, out);
                        rotT_vec(Rf, ww, out + 3);
                        for (int i = 0; i < dim; ++i) S.Jb[col][crow + i] += out[r0 + i];
                    } else {          // - rMf.toActionMatrixInverse() * reference frame Jacobian, LOCAL (frame.hpp:414-436)
                        T lv[3], lw[3];
                        cross3(pr, ww, pxw);
                        d[0] = v[0] - pxw[0]; d[1] = v[1] - pxw[1]; d[2] = v[2] - pxw[2];
                        rotT_vec(Rr, d, lv);
                        rotT_vec(Rr, ww, lw);
                        cross3(pm, lw, pxw);
                        d[0] = lv[0] - pxw[0]; d[1] = lv[1] - pxw[1]; d[2] = lv[2] - pxw[2];
                        rotT_vec(Rm, d, out);
                        rotT_vec(Rm, lw, out + 3);
                        for (int i = 0; i < dim; ++i) S.Jb[col][crow + i] -= out[r0 + i];
                    }
                }
            }
        }
        crow += dim;
    }
    cx.sync();
}

// dq <- dq - sum_r (w_r . dq) w_r over `rank` orthonormal rows of W (lane <-> column)
template <typename T, class Cfg, class Ctx>
IKB_HD void coop_project_out(const Ctx &cx, const T (*W)[Cfg::NV], int rank, int nv, T *dq) {
    constexpr int TEAM = Cfg::TEAM;
    const int lane = cx.lane;
    const int rounds = coop_warp_rounds(cx, rank);
    for (int r = 0; r < rounds; ++r) {
        const bool live = r < rank;
        T s = T(0);
        if (live)
            for (int c = lane; c < nv; c += TEAM) s += W[r][c] * dq[c];
        for (int off = TEAM / 2; off >= 1; off >>= 1) s += cx.shfl(s, lane ^ off);
        if (live)
            for (int c = lane; c < nv; c += TEAM) dq[c] -= s * W[r][c];
    }
    cx.sync();
}

// One iteration of ik::dls (dls.cpp:16-71) or ik::pik (pik.cpp:41-86) of one problem by its TEAM lanes.  Returns ||e[0]||^2
// (identical in all lanes).  Below `tol` the state is left untouched (dls.cpp:61-64), else q has been stepped and clamped.
template <typename T, class Cfg, bool SHFL, bool PIK, int EXTRA, class Ctx>
IKB_HD T coop_iteration(const Ctx &cx, const DevProblem<T> &P, CoopScratch<T, Cfg, EXTRA> &S, T step, T damping2, const T *pik_lambda2, T tol) {
    constexpr int TEAM = Cfg::TEAM, RPL = Cfg::RPL, M = Cfg::M;
    const int lane = cx.lane, nv = P.nv, rows = P.rows;
    coop_evaluate<T, Cfg, EXTRA>(cx, P, S);

    T res = T(0);
    for (int i = 0; i < P.rows_p0; ++i) res += S.e[i] * S.e[i];   // visitor.hpp:19

    if constexpr (!PIK) {
        T y[RPL];
        coop_gram_solve<T, Cfg, SHFL, Cfg::LD, false>(cx, S.Jt, P.col_rows, nv, S.e, rows, damping2, S.piv, y);
#pragma unroll
        for (int rr = 0; rr < RPL; ++rr) {
            const int r = lane + rr * TEAM;
            if (r < M) S.y[r] = y[rr];
        }
        cx.sync();
        for (int c = lane; c < nv; c += TEAM) {   // dq = -J^T y (dls.cpp:52)
            const T *col = S.Jt[c];
            T s = T(0);
            for (int r = 0; r < rows; ++r) s += col[r] * S.y[r];
            S.dq[c] = -s;
        }
        cx.sync();
        if constexpr (EXTRA >= 2) if (P.nconstraints > 0) {   // dq <- (I - Jc^+ Jc) dq (dls.cpp:26-34,44-52)
            coop_constraint_jacobian<T, Cfg, EXTRA>(cx, P, S);
            const int rank = coop_rowspace_basis<T, Cfg>(cx, S.Jb, P.crows, nv, S.W, S.y);
            coop_project_out<T, Cfg>(cx, S.W, rank, nv, S.dq);
        }
    } else {
        static_assert(EXTRA >= 2, "ik::pik needs the EXTRA = 2 scratch");
        // ik::pik step (pik.cpp:43-65): dq = 0, P = I; per priority level i: de = e_i - J_i dq; Jb = J_i P;
        // dq -= damp_pinv(Jb, lambda_i) de = Jb^T (Jb Jb^T + lambda_i^2 I)^-1 de; P -= pinv(Jb) Jb.  P is kept factored,
        // P = I - sum w w^T over the orthonormal row-space bases of the levels done so far (DESIGN.md 4.2).
        for (int c = lane; c < nv; c += TEAM) S.dq[c] = T(0);
        cx.sync();
        int nb = 0, last_lvl = 0, row0 = 0;
        for (int lvl = 0; lvl < P.nlevels; ++lvl)
            if (P.level_rows[lvl] > 0) last_lvl = lvl;
        for (int lvl = 0; lvl < P.nlevels; ++lvl) {
            const int mi = P.level_rows[lvl];
            if (mi == 0) continue;
            // lane <-> level row: de_bar (pik.cpp:49) and Jbar = J_i P (pik.cpp:51); rows >= mi of Jb are zeroed
            for (int r = lane; r < Cfg::LDX; r += TEAM) {
                if (r < mi) {
                    T s = T(0);
                    for (int c = 0; c < nv; ++c) {
                        const T jrc = S.Jt[c][row0 + r];
                        s += jrc * S.dq[c];
                        S.Jb[c][r] = jrc;
                    }
                    S.y[r] = S.e[row0 + r] - s;
                    for (int k = 0; k < nb; ++k) {
                        T t = T(0);
                        for (int c = 0; c < nv; ++c) t += S.Jt[c][row0 + r] * S.W[k][c];
                        for (int c = 0; c < nv; ++c) S.Jb[c][r] -= t * S.W[k][c];
                    }
                } else {
                    for (int c = 0; c < nv; ++c) S.Jb[c][r] = T(0);
                    if (r < M + 2) S.y[r] = T(0);
                }
            }
            cx.sync();
            T z[RPL];
            coop_gram_solve<T, Cfg, SHFL, Cfg::LDX, true>(cx, S.Jb, (const uint64_t *)nullptr, nv, S.y, mi, pik_lambda2[lvl], S.piv, z);
            cx.sync();   // everybody has read the right-hand side from S.y
#pragma unroll
            for (int rr = 0; rr < RPL; ++rr) {
                const int r = lane + rr * TEAM;
                if (r < M) S.y[r] = z[rr];
            }
            cx.sync();
            for (int c = lane; c < nv; c += TEAM) {   // dq -= Jb^T z (pik.cpp:54-55)
                const T *col = S.Jb[c];
                T s = T(0);
                for (int r = 0; r < mi; ++r) s += col[r] * S.y[r];
                S.dq[c] -= s;
            }
            cx.sync();
            if (lvl != last_lvl) nb += coop_rowspace_basis<T, Cfg>(cx, S.Jb, mi, nv, S.W + nb, S.y);
            row0 += mi;
        }
    }

    if (!(res < tol)) {   // dls.cpp:61-71
        for (int j = 1 + lane; j < P.njoints; j += TEAM) {
            const int iq = P.idx_q[j], iv = P.idx_v[j], jt = P.jtype[j];
            if (jt == IKB_J_FREEFLYER) {
                T v6[6], R0[9];
                for (int i = 0; i < 6; ++i) v6[i] = step * S.dq[iv + i];
                quat_to_rot(S.q[iq + 3], S.q[iq + 4], S.q[iq + 5], S.q[iq + 6], R0);
                integrate_freeflyer(R0, &S.q[iq], &S.q[iq + 3], v6);
                for (int k = 0; k < 7; ++k) S.q[iq + k] = min_(P.upper[iq + k], max_(S.q[iq + k], P.lower[iq + k]));
            } else if (is_continuous(jt)) {   // SpecialOrthogonalOperation<2>::integrate: rotate (c, s) by the step, first-order renormalisation
                T sw, cw;
                sincos_(step * S.dq[iv], &sw, &cw);
                const T c0 = S.q[iq], s0 = S.q[iq + 1];
                const T c1 = cw * c0 - sw * s0, s1 = sw * c0 + cw * s0;
                const T a = (T(3) - (c1 * c1 + s1 * s1)) / T(2);
                S.q[iq] = min_(P.upper[iq], max_(c1 * a, P.lower[iq]));
                S.q[iq + 1] = min_(P.upper[iq + 1], max_(s1 * a, P.lower[iq + 1]));
            } else {
                S.q[iq] = min_(P.upper[iq], max_(S.q[iq] + step * S.dq[iv], P.lower[iq]));
            }
        }
    }
    cx.sync();
    return res;
}

// Once per kernel (per team): the structural zeros and the constant entries of J.
template <typename T, class Cfg, int EXTRA, class Ctx> IKB_HD void coop_init_scratch(const Ctx &cx, const DevProblem<T> &P, CoopScratch<T, Cfg, EXTRA> &S) {
    constexpr int TEAM = Cfg::TEAM;
    T *z = &S.Jt[0][0];
    for (int i = cx.lane; i < Cfg::NV * Cfg::LD; i += TEAM) z[i] = T(0);
    for (int i = cx.lane; i < Cfg::M + 2; i += TEAM) { S.e[i] = T(0); S.y[i] = T(0); }
    for (int i = cx.lane; i < Cfg::NQ; i += TEAM) S.q[i] = T(0);
    for (int i = cx.lane; i < Cfg::TSZ; i += TEAM) S.tg[i] = (i % 12 == 0 || i % 12 == 4 || i % 12 == 8) ? T(1) : T(0);
    cx.sync();
    if (cx.lane == 0) {
        for (int i = 0; i < 12; ++i) S.oM[0][i] = (i % 4 == 0 && i < 9) ? T(1) : T(0);   // joint 0 = universe: identity, never recomputed
        for (int j = 1; j < P.njoints; ++j)
            if (P.jtype[j] == IKB_J_FREEFLYER) S.q[P.idx_q[j] + 6] = T(1);   // a team without a problem iterates on the neutral pose
            else if (is_continuous(P.jtype[j])) S.q[P.idx_q[j]] = T(1);
        for (int t = 0; t < P.ntasks; ++t)
            if (P.t_kind[t] == IKB_TASK_POSTURE) {   // posture.hpp:60-66: J.rightCols(nj) = I (not masked), weighted (data.cpp:50)
                const int nj = P.t_type[t], row = P.t_row[t];
                for (int i = 0; i < nj; ++i) S.Jt[P.nv - nj + i][row + i] = P.weight[row + i];
            }
    }
    cx.sync();
}

#if defined(__CUDACC__)
template <int TEAM> struct CoopDevCtx {
    int lane;
    __device__ __forceinline__ void sync() const { __syncwarp(); }
    __device__ __forceinline__ int warp_max(int v) const { return __reduce_max_sync(0xffffffffu, v); }
    __device__ __forceinline__ double shfl(double v, int src) const { return __shfl_sync(0xffffffffu, v, src, TEAM); }
    __device__ __forceinline__ float shfl(float v, int src) const { return __shfl_sync(0xffffffffu, v, src, TEAM); }
};

template <typename T, class Cfg, int EXTRA> struct CoopLaunch {
    static constexpr size_t kBlob = (sizeof(DevProblem<T>) + 15) / 16 * 16 + 16;   // + mbarrier
    static constexpr size_t kScratch = sizeof(CoopScratch<T, Cfg, EXTRA>);
    static constexpr int kTeamsPerWarp = 32 / Cfg::TEAM;
    // one CTA per SM, as many teams as shared memory and a 128-register budget per thread allow
    static constexpr int kBySmem = (int)((227 * 1024 - kBlob) / kScratch);
    static constexpr int kWarps0 = kBySmem / kTeamsPerWarp < 16 ? kBySmem / kTeamsPerWarp : 16;
    static constexpr int kWarps = kWarps0 < 1 ? 1 : kWarps0;
    static constexpr int kTeams = kWarps * kTeamsPerWarp;
    static constexpr int kThreads = kWarps * 32;
    static constexpr size_t kSmem = kBlob + (size_t)kTeams * kScratch;
    static_assert(kBlob + kTeamsPerWarp * kScratch <= 227 * 1024, "one warp of teams must fit in shared memory");
};

__device__ __forceinline__ void coop_stage_blob(void *smem_dst, const void *gmem_src, unsigned bytes, unsigned long long *bar) {
    // TMA bulk copy of the constant blob (URDF constants + tables) into shared memory, once per CTA
    const unsigned bar_addr = (unsigned)__cvta_generic_to_shared(bar);
    const unsigned dst_addr = (unsigned)__cvta_generic_to_shared(smem_dst);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_addr));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_addr), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_addr),
                     "l"(gmem_src), "r"(bytes), "r"(bar_addr)
                     : "memory");
    }
    unsigned done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar_addr)
            : "memory");
    }
}

// Persistent teams; every team pulls problem indices from a global ticket counter (as dls_team.cuh).
template <typename T, class Cfg, bool SHFL, bool PIK, int EXTRA>
__global__ void __launch_bounds__(CoopLaunch<T, Cfg, EXTRA>::kThreads, 1) dls_coop_kernel(const DevProblem<T> *__restrict__ gP, const __grid_constant__ SolveArgs<T> a) {
    using L = CoopLaunch<T, Cfg, EXTRA>;
    constexpr int TEAM = Cfg::TEAM;
    extern __shared__ __align__(16) unsigned char coop_smem[];
    DevProblem<T> &P = *reinterpret_cast<DevProblem<T> *>(coop_smem);
    unsigned long long *bar = reinterpret_cast<unsigned long long *>(coop_smem + L::kBlob - 16);
    coop_stage_blob(&P, gP, (unsigned)sizeof(DevProblem<T>), bar);
    const int lane = threadIdx.x & (TEAM - 1), team = threadIdx.x / TEAM;
    CoopScratch<T, Cfg, EXTRA> &S = reinterpret_cast<CoopScratch<T, Cfg, EXTRA> *>(coop_smem + L::kBlob)[team];
    const CoopDevCtx<TEAM> cx{lane};
    coop_init_scratch<T, Cfg, EXTRA>(cx, P, S);

    const int nq = P.nq, tsz = P.tsz;
    long long b = 0;
    int it = 0;
    bool have = false, need = true, first = true;
    // The first ticket of a team is static and strided over the CTAs (team t of CTA c starts with problem t * gridDim + c),
    // so a batch smaller than the grid spreads over all SMs instead of filling the first CTAs; later tickets come from the
    // global counter, offset by the number of static ones.
    const unsigned long long n_static = (unsigned long long)gridDim.x * L::kTeams;
    for (;;) {
        unsigned long long t = 0;
        if (need && !first && lane == 0) t = atomicAdd(a.ticket, 1ULL) + n_static;
        t = __shfl_sync(0xffffffffu, t, 0, TEAM);
        if (need) {
            if (first) t = (unsigned long long)team * gridDim.x + blockIdx.x;
            first = false;
            it = 0;
            have = (long long)t < a.B;
            b = (long long)t;
            if (have) {
                const T *qb = a.q0 + b * a.q0_bs;
                for (int k = lane; k < nq; k += TEAM) S.q[k] = qb[k * a.q0_es];
                const T *tb = a.targets + b * a.tg_bs;
                for (int k = lane; k < tsz; k += TEAM) S.tg[k] = tb[k * a.tg_es];
            }
            need = false;
        }
        // Warps run free of each other.  (Measured: a CTA-wide barrier per trip, which lets the warps share the ~85 KB of
        // SASS they stream per iteration, takes `no_instruction` from 1.42 to 0.13 stalls per issue but costs 0.93 in
        // barrier stalls, +1.0 in shared-memory scoreboard stalls -- every warp hits the same phase at once -- and +25 %
        // executed instructions from teams idling in step: 3.31 -> 3.54 ms on 65 536 Cassie problems, profiles/r2_coop_*.)
        __syncwarp();
        if (!__any_sync(0xffffffffu, have)) break;

        const T res = coop_iteration<T, Cfg, SHFL, PIK, EXTRA>(cx, P, S, a.step_length, a.damping2, a.pik_lambda2, a.tolerance);

        if (have) {
            const bool converged = res < a.tolerance;       // visitor.hpp:19
            if (!converged) ++it;
            if (converged || it >= a.max_iterations) {      // dls.cpp:61-64 / 14,76-77
                T *qo = a.q + b * a.q_bs;
                for (int k = lane; k < nq; k += TEAM) qo[k * a.q_es] = S.q[k];
                if (lane == 0) {
                    if (a.success) a.success[b] = converged ? 1 : 0;
                    if (a.iters) a.iters[b] = it;
                    if (a.resid) a.resid[b] = res;
                }
                // *_solve_ex: what the reference leaves in dls_data after the call (data.hpp:15-28) -- dq, e, J of the LAST evaluation
                const int nv = P.nv, rows = P.rows;
                if (a.aux_dq) for (int c = lane; c < nv; c += TEAM) a.aux_dq[b * nv + c] = S.dq[c];
                if (a.aux_e) for (int r = lane; r < rows; r += TEAM) a.aux_e[b * rows + r] = S.e[r];
                if (a.aux_J) for (int i = lane; i < rows * nv; i += TEAM) a.aux_J[(long long)b * rows * nv + i] = S.Jt[i % nv][i / nv];
                need = true;
                have = false;
            }
        }
    }
}
#endif  // __CUDACC__

}  // namespace ikb
