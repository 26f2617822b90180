// Generic (table-driven) batched DLS IK kernel: any tree topology / task list that fits the capacity
// template parameters.  One IK problem per THREAD, the whole ik::dls loop (reference dls.cpp:14-74) runs
// in-kernel: FK (data.cpp:28-29) -> frame Jacobians (data.cpp:30, frame.hpp:169-170) -> SE3 log error +
// Jlog6 (frame.hpp:37-62,152-182) -> weighting (data.cpp:49-50) -> Gram + damping (dls.cpp:39-41) ->
// LDL^T solve and dq = -J^T y (dls.cpp:52-53) -> stop test (visitor.hpp:19) -> integrate (dls.cpp:67-68)
// -> clamp (common.hpp:53-56).
//
// This is the correctness baseline and the fallback for arbitrary robots: per-problem scratch (joint
// placements, J, Gram) lives in per-thread local memory and is indexed dynamically from the tables in the
// shared-memory problem blob.  The specialised kernels (dls_*.cu) are the fast path.
//
// Scheduling: lanes pull problem indices from a global ticket counter; a lane whose problem finishes
// (converged or out of iterations) immediately loads the next one, so every lane of a warp executes the
// same evaluate/solve body each trip regardless of how iteration counts differ across problems
// (median 4, p95 13, max 100 on the Cassie workload; SURVEY.md 6).
#pragma once
#include <cuda_runtime.h>

#include "dev_problem.hpp"
#include "joint_types.hpp"
#include "se3_math.cuh"

namespace ikb {

// ---- TMA bulk copy of the constant blob into shared memory ---------------------------------------------
__device__ __forceinline__ void stage_blob_tma(void *smem_dst, const void *gmem_src, unsigned bytes,
                                               unsigned long long *bar) {
    const unsigned bar_addr = (unsigned)__cvta_generic_to_shared(bar);
    const unsigned dst_addr = (unsigned)__cvta_generic_to_shared(smem_dst);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_addr));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_addr), "r"(bytes) : "memory");
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_addr),
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

// unit axis of a revolute, continuous or prismatic joint in its own frame
template <typename T>
__device__ __forceinline__ void joint_axis_local(const DevProblem<T> &P, int j, T *a) {
    const int t = as_revolute(P.jtype[j]);
    a[0] = a[1] = a[2] = T(0);
    if (t == IKB_J_RX || t == IKB_J_PX) a[0] = 1;
    else if (t == IKB_J_RY || t == IKB_J_PY) a[1] = 1;
    else if (t == IKB_J_RZ || t == IKB_J_PZ) a[2] = 1;
    else { a[0] = P.axis[j][0]; a[1] = P.axis[j][1]; a[2] = P.axis[j][2]; }
}

// joint transform liMi = placement * M_j(q) for every joint type the flattener emits
template <typename T>
__device__ __forceinline__ void joint_local(const DevProblem<T> &P, int j, const T *q, T *Rl, T *pl) {
    const T *PR = P.placement[j], *Pp = PR + 9;
    const int t = P.jtype[j];
    const T *qj = q + P.idx_q[j];
    if (t == IKB_J_FREEFLYER) {
        T Rj[9];
        quat_to_rot(qj[3], qj[4], qj[5], qj[6], Rj);
        se3_mul(PR, Pp, Rj, qj, Rl, pl);
    } else if (is_revolute_like(t)) {
        T s, c, Rj[9];
        if (is_continuous(t)) { c = qj[0]; s = qj[1]; }   // (cos, sin) as given, not renormalised (RevoluteUnbounded::calc)
        else sincos_(qj[0], &s, &c);
        const int r = as_revolute(t);
        if (r == IKB_J_RX) {
            Rj[0] = 1; Rj[1] = 0; Rj[2] = 0; Rj[3] = 0; Rj[4] = c; Rj[5] = -s; Rj[6] = 0; Rj[7] = s; Rj[8] = c;
        } else if (r == IKB_J_RY) {
            Rj[0] = c; Rj[1] = 0; Rj[2] = s; Rj[3] = 0; Rj[4] = 1; Rj[5] = 0; Rj[6] = -s; Rj[7] = 0; Rj[8] = c;
        } else if (r == IKB_J_RZ) {
            Rj[0] = c; Rj[1] = -s; Rj[2] = 0; Rj[3] = s; Rj[4] = c; Rj[5] = 0; Rj[6] = 0; Rj[7] = 0; Rj[8] = 1;
        } else {
            const T *a = P.axis[j];
            const T v = 1 - c;
            Rj[0] = a[0] * a[0] * v + c;        Rj[1] = a[0] * a[1] * v - a[2] * s; Rj[2] = a[0] * a[2] * v + a[1] * s;
            Rj[3] = a[0] * a[1] * v + a[2] * s; Rj[4] = a[1] * a[1] * v + c;        Rj[5] = a[1] * a[2] * v - a[0] * s;
            Rj[6] = a[0] * a[2] * v - a[1] * s; Rj[7] = a[1] * a[2] * v + a[0] * s; Rj[8] = a[2] * a[2] * v + c;
        }
        mat3_mul(PR, Rj, Rl);
        pl[0] = Pp[0]; pl[1] = Pp[1]; pl[2] = Pp[2];
    } else {  // prismatic
        T a[3] = {T(0), T(0), T(0)};
        if (t == IKB_J_PX) a[0] = 1;
        else if (t == IKB_J_PY) a[1] = 1;
        else if (t == IKB_J_PZ) a[2] = 1;
        else { a[0] = P.axis[j][0]; a[1] = P.axis[j][1]; a[2] = P.axis[j][2]; }
        T d[3] = {a[0] * qj[0], a[1] * qj[0], a[2] * qj[0]}, o[3];
        rot_vec(PR, d, o);
#pragma unroll
        for (int i = 0; i < 9; ++i) Rl[i] = PR[i];
        pl[0] = Pp[0] + o[0]; pl[1] = Pp[1] + o[1]; pl[2] = Pp[2] + o[2];
    }
}

// Forward kinematics of every joint (world placements), oR/op indexed by joint; joint 0 = universe = identity.
template <typename T, int NJ>
__device__ __forceinline__ void fk_all(const DevProblem<T> &P, const T *q, T (*oR)[9], T (*op)[3]) {
#pragma unroll
    for (int i = 0; i < 9; ++i) oR[0][i] = (i % 4 == 0) ? T(1) : T(0);
    op[0][0] = op[0][1] = op[0][2] = T(0);
    for (int j = 1; j < P.njoints; ++j) {
        T Rl[9], pl[3];
        joint_local(P, j, q, Rl, pl);
        const int par = P.parent[j];
        se3_mul(oR[par], op[par], Rl, pl, oR[j], op[j]);
    }
}

// Orthonormal basis W (rank rows) of the row space of the numerically rank-r part of A (mi x nv, destroyed): what
// A.completeOrthogonalDecomposition().pseudoInverse() * A projects onto (pik.cpp:59-61, dls.cpp:44-49).  Householder QR with
// column pivoting in place, r from Eigen's threshold eps * min(m, n) * max pivot, the first r rows of R (columns back in
// place) orthonormalised by modified Gram-Schmidt, twice.  `diag` is scratch for mi scalars.
template <typename T, int NV, int MR>
__device__ __forceinline__ int rowspace_basis(T (*A)[NV], int mi, int nv, T (*W)[NV], T *diag) {
    int perm[NV];
    for (int c = 0; c < nv; ++c) perm[c] = c;
    const int steps = mi < nv ? mi : nv;
    T maxpiv = T(0);
    for (int k = 0; k < steps; ++k) {
        int best = k;
        T bn = T(-1);
        for (int c = k; c < nv; ++c) {
            T s = T(0);
            for (int r = k; r < mi; ++r) s += A[r][c] * A[r][c];
            if (s > bn) { bn = s; best = c; }
        }
        if (best != k) {
            for (int r = 0; r < mi; ++r) { const T t = A[r][k]; A[r][k] = A[r][best]; A[r][best] = t; }
            const int t = perm[k]; perm[k] = perm[best]; perm[best] = t;
        }
        const T nrm = sqrt_(max_(bn, T(0)));
        if (!(nrm > T(0))) { diag[k] = T(0); continue; }
        const T alpha = A[k][k] >= T(0) ? -nrm : nrm;
        T v[MR];
        T vn = T(0);
        for (int r = k; r < mi; ++r) v[r] = A[r][k];
        v[k] -= alpha;
        for (int r = k; r < mi; ++r) vn += v[r] * v[r];
        if (vn > T(0)) {
            const T two_over = T(2) / vn;
            for (int c = k; c < nv; ++c) {
                T s = T(0);
                for (int r = k; r < mi; ++r) s += v[r] * A[r][c];
                s *= two_over;
                for (int r = k; r < mi; ++r) A[r][c] -= s * v[r];
            }
        }
        diag[k] = abs_(A[k][k]);
        maxpiv = max_(maxpiv, diag[k]);
    }
    const T eps = sizeof(T) == 8 ? T(2.220446049250313e-16) : T(1.1920929e-7);
    const T thr = eps * T(steps) * maxpiv;
    int rank = 0;
    for (int k = 0; k < steps; ++k) rank += diag[k] > thr ? 1 : 0;
    for (int r = 0; r < rank; ++r)
        for (int c = 0; c < nv; ++c) W[r][perm[c]] = c >= r ? A[r][c] : T(0);
    for (int pass = 0; pass < 2; ++pass)
        for (int r = 0; r < rank; ++r) {
            for (int p2 = 0; p2 < r; ++p2) {
                T s = T(0);
                for (int c = 0; c < nv; ++c) s += W[r][c] * W[p2][c];
                for (int c = 0; c < nv; ++c) W[r][c] -= s * W[p2][c];
            }
            T nr = T(0);
            for (int c = 0; c < nv; ++c) nr += W[r][c] * W[r][c];
            const T inr = T(1) / sqrt_(nr);
            for (int c = 0; c < nv; ++c) W[r][c] *= inr;
        }
    return rank;
}

// World column (linear v, angular w) of velocity coordinate cc of joint j (data.cpp:30: oMi.act(S_i)).
template <typename T, int NJ>
__device__ __forceinline__ void world_column(const DevProblem<T> &P, int j, int cc, const T (*oR)[9], const T (*op)[3], T *v, T *ww) {
    const int jt = P.jtype[j];
    if (jt == IKB_J_FREEFLYER) {
        const int ax = cc % 3;
        const T rc[3] = {oR[j][ax], oR[j][3 + ax], oR[j][6 + ax]};
        if (cc < 3) { v[0] = rc[0]; v[1] = rc[1]; v[2] = rc[2]; ww[0] = ww[1] = ww[2] = T(0); }
        else { cross3(op[j], rc, v); ww[0] = rc[0]; ww[1] = rc[1]; ww[2] = rc[2]; }
    } else {
        T al[3], z[3];
        joint_axis_local(P, j, al);
        rot_vec(oR[j], al, z);
        if (is_revolute_like(jt)) { cross3(op[j], z, v); ww[0] = z[0]; ww[1] = z[1]; ww[2] = z[2]; }
        else { v[0] = z[0]; v[1] = z[1]; v[2] = z[2]; ww[0] = ww[1] = ww[2] = T(0); }
    }
}

// PIK = false: ik::dls (dls.cpp:5-78).  PIK = true: ik::pik (pik.cpp:31-96) -- same evaluate / stop test / integrate, the
// step comes from the priority recursion below instead of one damped solve of the stacked system.
template <typename T, int NJ, int NV, int M, bool PIK = false>
__global__ void __launch_bounds__(128) dls_generic_kernel(const DevProblem<T> *__restrict__ gP, SolveArgs<T> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DevProblem<T> &P = *reinterpret_cast<DevProblem<T> *>(smem_raw);
    unsigned long long *bar = reinterpret_cast<unsigned long long *>(smem_raw + sizeof(DevProblem<T>));
    stage_blob_tma(&P, gP, (unsigned)sizeof(DevProblem<T>), bar);

    constexpr int NQ = NV + 4;
    T q[NQ];
    T oR[NJ][9], op[NJ][3];
    T J[M][NV], e[M], y[M], G[M * (M + 1) / 2], dq[NV];

    const int nq = P.nq, nv = P.nv, rows = P.rows;
    // Work fetch.  First launch: tickets are problem indices.  Second launch of a two-phase solve (a.resume): tickets
    // index the list of problems the first one suspended after a.it_cap steps; they continue from their saved iterate.
    // (Why two launches: a straggler alone in its warp touches one 4-byte word per 128-byte line of local memory, so
    // its ~8 KB of scratch occupy a whole L1; compacted 32 to a warp the stragglers run from L1 -- DESIGN.md 4.2.)
    long long b = 0;
    bool have = false;
    int it = 0;
    auto fetch = [&]() {
        b = (long long)atomicAdd(a.ticket, 1ULL);
        if (!a.resume) {
            have = b < a.B;
            it = 0;
            if (have)
                for (int k = 0; k < nq; ++k) q[k] = a.q0[k * a.q0_es + b * a.q0_bs];
        } else {
            have = b < (long long)*a.list_count;
            if (have) {
                b = a.list[b];
                it = a.iters_ws[b];
                for (int k = 0; k < nq; ++k) q[k] = a.q[k * a.q_es + b * a.q_bs];
            }
        }
    };
    fetch();

    while (__any_sync(0xffffffffu, have)) {
        if (have) {
            // ---- evaluate_problem_data ----
            fk_all<T, NJ>(P, q, oR, op);
            for (int r = 0; r < rows; ++r)
                for (int c = 0; c < nv; ++c) J[r][c] = T(0);
            for (int t = 0; t < P.ntasks; ++t) {
                const int row = P.t_row[t], dim = P.t_dim[t], kind = P.t_kind[t];
                const T *tg = a.targets + b * a.tg_bs;
                const long long es = a.tg_es;
                const int toff = P.t_toff[t];
                if (kind == IKB_TASK_POSTURE) {
                    const int nj = P.t_type[t];
                    for (int i = 0; i < nj; ++i) {
                        e[row + i] = (q[nq - nj + i] - tg[(toff + i) * es]) * P.mask[P.t_moff[t] + i];
                        J[row + i][nv - nj + i] = T(1);
                    }
                } else if (kind == IKB_TASK_COM) {
                    // CentreOfMassTask (centre_of_mass.hpp:24-38, data.cpp:31-34): backward pass accumulating the mass and
                    // first moment of every subtree (joints are stored parents first), e = oMr^-1 com - target, and per
                    // velocity coordinate the velocity it gives its subtree's centre of mass, weighted by the subtree's
                    // share of the total mass, rotated into the reference frame (which the reference does not differentiate).
                    T ms[NJ], mc[NJ][3];
                    for (int j = 1; j < P.njoints; ++j) {
                        T cw[3];
                        rot_vec(oR[j], P.com[j], cw);
                        ms[j] = P.mass[j];
                        for (int i = 0; i < 3; ++i) mc[j][i] = P.mass[j] * (cw[i] + op[j][i]);
                    }
                    T tot[3] = {T(0), T(0), T(0)};
                    for (int j = P.njoints - 1; j >= 1; --j) {
                        const int par = P.parent[j];
                        if (par > 0) {
                            ms[par] += ms[j];
                            for (int i = 0; i < 3; ++i) mc[par][i] += mc[j][i];
                        } else {
                            for (int i = 0; i < 3; ++i) tot[i] += mc[j][i];
                        }
                    }
                    const T inv_m = T(1) / P.total_mass;
                    const int r = P.t_ref[t], rj = P.f_parent[r];
                    T Rr[9], pr[3], d[3], lc[3];
                    se3_mul(oR[rj], op[rj], P.f_placement[r], P.f_placement[r] + 9, Rr, pr);
                    for (int i = 0; i < 3; ++i) d[i] = tot[i] * inv_m - pr[i];
                    rotT_vec(Rr, d, lc);
                    for (int i = 0; i < 3; ++i) e[row + i] = lc[i] - tg[(toff + i) * es];
                    for (int j = 1; j < P.njoints; ++j) {
                        if (!(ms[j] > T(0))) continue;
                        const T share = ms[j] * inv_m, ims = T(1) / ms[j];
                        const T cs[3] = {mc[j][0] * ims, mc[j][1] * ims, mc[j][2] * ims};
                        const int ncol = P.jtype[j] == IKB_J_FREEFLYER ? 6 : 1;
                        for (int cc = 0; cc < ncol; ++cc) {
                            T v[3], ww[3], wxc[3], vel[3];
                            world_column<T, NJ>(P, j, cc, oR, op, v, ww);
                            cross3(ww, cs, wxc);
                            for (int i = 0; i < 3; ++i) vel[i] = share * (v[i] + wxc[i]);
                            rotT_vec(Rr, vel, lc);
                            for (int i = 0; i < 3; ++i) J[row + i][P.idx_v[j] + cc] = lc[i];
                        }
                    }
                } else {
                    const int f = P.t_frame[t], r = P.t_ref[t];
                    const int fj = P.f_parent[f], rj = P.f_parent[r];
                    T Rf[9], pf[3], Rr[9], pr[3];
                    se3_mul(oR[fj], op[fj], P.f_placement[f], P.f_placement[f] + 9, Rf, pf);
                    se3_mul(oR[rj], op[rj], P.f_placement[r], P.f_placement[r] + 9, Rr, pr);
                    if (kind == IKB_TASK_FRAME) {
                        T Rt[9], pt[3], Rtg[9], ptg[3];
#pragma unroll
                        for (int i = 0; i < 9; ++i) Rtg[i] = tg[(toff + i) * es];
#pragma unroll
                        for (int i = 0; i < 3; ++i) ptg[i] = tg[(toff + 9 + i) * es];
                        se3_mul(Rr, pr, Rtg, ptg, Rt, pt);  // oMt = oMr * target
                        // error: log6(fMt)
                        T Re[9], pe[3], w[3], th, sth, cth, lin[3];
                        se3_actinv(Rf, pf, Rt, pt, Re, pe);
                        log3(Re, w, th, sth, cth);
                        LogCoeffs<T> lc = log_coeffs(th, sth, cth);
                        log6_from(w, lc, pe, lin);
                        const int ktype = P.t_type[t];
                        if (ktype == IKB_POSITION) { e[row] = lin[0]; e[row + 1] = lin[1]; e[row + 2] = lin[2]; }
                        else if (ktype == IKB_ORIENTATION) { e[row] = w[0]; e[row + 1] = w[1]; e[row + 2] = w[2]; }
                        else {
                            e[row] = lin[0]; e[row + 1] = lin[1]; e[row + 2] = lin[2];
                            e[row + 3] = w[0]; e[row + 4] = w[1]; e[row + 5] = w[2];
                        }
                        // Jacobian: rows of -Jlog6(tMf) * Jf_LOCAL
                        T Rm[9], pm[3], w2[3], th2, sth2, cth2, A[9], Bm[9];
                        se3_actinv(Rt, pt, Rf, pf, Rm, pm);
                        log3(Rm, w2, th2, sth2, cth2);
                        LogCoeffs<T> lc2 = log_coeffs(th2, sth2, cth2);
                        jlog6_blocks(w2, th2, lc2, pm, A, Bm);
                        for (int j = fj; j > 0; j = P.parent[j]) {
                            const int c0 = P.idx_v[j], jt = P.jtype[j];
                            const int ncol = jt == IKB_J_FREEFLYER ? 6 : 1;
                            for (int cc = 0; cc < ncol; ++cc) {
                                T v[3], ww[3];
                                if (jt == IKB_J_FREEFLYER) {
                                    const int ax = cc % 3;
                                    T rc[3] = {oR[j][ax], oR[j][3 + ax], oR[j][6 + ax]};
                                    if (cc < 3) { v[0] = rc[0]; v[1] = rc[1]; v[2] = rc[2]; ww[0] = ww[1] = ww[2] = T(0); }
                                    else { cross3(op[j], rc, v); ww[0] = rc[0]; ww[1] = rc[1]; ww[2] = rc[2]; }
                                } else {
                                    T al[3], z[3];
                                    joint_axis_local(P, j, al);
                                    rot_vec(oR[j], al, z);
                                    if (is_revolute_like(jt)) { cross3(op[j], z, v); ww[0] = z[0]; ww[1] = z[1]; ww[2] = z[2]; }
                                    else { v[0] = z[0]; v[1] = z[1]; v[2] = z[2]; ww[0] = ww[1] = ww[2] = T(0); }
                                }
                                // oMf.actInv(column)
                                T pxw[3], d[3], lv[3], lw[3];
                                cross3(pf, ww, pxw);
                                d[0] = v[0] - pxw[0]; d[1] = v[1] - pxw[1]; d[2] = v[2] - pxw[2];
                                rotT_vec(Rf, d, lv);
                                rotT_vec(Rf, ww, lw);
                                T top[3], bot[3];
#pragma unroll
                                for (int i = 0; i < 3; ++i) {
                                    top[i] = -(A[3 * i] * lv[0] + A[3 * i + 1] * lv[1] + A[3 * i + 2] * lv[2] +
                                               Bm[3 * i] * lw[0] + Bm[3 * i + 1] * lw[1] + Bm[3 * i + 2] * lw[2]);
                                    bot[i] = -(A[3 * i] * lw[0] + A[3 * i + 1] * lw[1] + A[3 * i + 2] * lw[2]);
                                }
                                const int c = c0 + cc;
                                if (ktype == IKB_POSITION) { J[row][c] = top[0]; J[row + 1][c] = top[1]; J[row + 2][c] = top[2]; }
                                else if (ktype == IKB_ORIENTATION) { J[row][c] = bot[0]; J[row + 1][c] = bot[1]; J[row + 2][c] = bot[2]; }
                                else {
                                    J[row][c] = top[0]; J[row + 1][c] = top[1]; J[row + 2][c] = top[2];
                                    J[row + 3][c] = bot[0]; J[row + 4][c] = bot[1]; J[row + 5][c] = bot[2];
                                }
                            }
                        }
                    } else {  // IKB_TASK_ALIGN_AXIS (frame.hpp:246-299)
                        T Rm[9], pm[3];
                        se3_actinv(Rr, pr, Rf, pf, Rm, pm);  // rMf
                        const int ax = P.t_type[t];
                        T rv[3] = {Rm[ax], Rm[3 + ax], Rm[6 + ax]};
                        T tn[3] = {tg[toff * es], tg[(toff + 1) * es], tg[(toff + 2) * es]};
                        const T n = sqrt_(dot3(tn, tn));
                        tn[0] /= n; tn[1] /= n; tn[2] /= n;
                        e[row] = T(1) - dot3(rv, tn);
                        T rxt[3], r3[3];
                        cross3(rv, tn, rxt);
                        rotT_vec(Rm, rxt, r3);  // (r x t)^T R_rMf
                        for (int j = fj; j > 0; j = P.parent[j]) {
                            const int c0 = P.idx_v[j], jt = P.jtype[j];
                            if (is_prismatic(jt)) continue;  // no angular part
                            const int ncol = jt == IKB_J_FREEFLYER ? 6 : 1;
                            for (int cc = (jt == IKB_J_FREEFLYER ? 3 : 0); cc < ncol; ++cc) {
                                T ww[3];
                                if (jt == IKB_J_FREEFLYER) {
                                    const int k = cc - 3;
                                    ww[0] = oR[j][k]; ww[1] = oR[j][3 + k]; ww[2] = oR[j][6 + k];
                                } else {
                                    T al[3];
                                    joint_axis_local(P, j, al);
                                    rot_vec(oR[j], al, ww);
                                }
                                T lw[3];
                                rotT_vec(Rf, ww, lw);
                                J[row][c0 + cc] = -dot3(r3, lw);
                            }
                        }
                    }
                }
                // weighting (data.cpp:49-50)
                for (int i = 0; i < dim; ++i) {
                    const T wgt = P.weight[row + i];
                    if (wgt != T(1)) {  // Task::weighting() defaults to ones (task.hpp:48-51)
                        e[row + i] *= wgt;
                        for (int c = 0; c < nv; ++c) J[row + i][c] *= wgt;
                    }
                }
            }
            if constexpr (PIK) {
                // ---- ik::pik step (pik.cpp:43-65): dq = 0, P = I; for every priority level i:
                //        de = e_i - J_i dq;  Jb = J_i P;  dq -= damp_pinv(Jb, lambda_i) de;  P -= pinv(Jb) Jb
                //      damp_pinv(Jb, l) = sum s/(l^2+s^2) v u^T (pik.cpp:5-21) == Jb^T (Jb Jb^T + l^2 I)^-1, so the damped
                //      step is one LDL^T solve; pinv(Jb) Jb (Eigen COD, pik.cpp:59-61) is the projector onto the row space
                //      of the numerically rank-r part of Jb: Householder QR with column pivoting, rank from Eigen's
                //      threshold eps * min(m, n) * max pivot, rows orthonormalised (modified Gram-Schmidt, twice). ----
                // The projector is kept factored, P = I - sum_k w_k w_k^T, with the orthonormal row-space bases w of the
                // levels done so far (each level's Jb = J_i P lies in range(P), so its basis is orthogonal to the earlier
                // ones): Jb = J_i - (J_i W^T) W costs rows x basis x nv instead of rows x nv x nv, the first level (P = I) is
                // free, the last level's update is never read, and the nv x nv matrix leaves the per-thread scratch.
                T Wall[M][NV];
                int nb = 0, last_lvl = 0;
                for (int i = 0; i < nv; ++i) dq[i] = T(0);
                for (int lvl = 0; lvl < P.nlevels; ++lvl)
                    if (P.level_rows[lvl] > 0) last_lvl = lvl;
                int row0 = 0;
                for (int lvl = 0; lvl < P.nlevels; ++lvl) {
                    const int mi = P.level_rows[lvl];
                    if (mi == 0) continue;
                    T Jb[M][NV];
                    for (int r = 0; r < mi; ++r) {
                        T s = T(0);
                        for (int c = 0; c < nv; ++c) {
                            const T jrc = J[row0 + r][c];
                            s += jrc * dq[c];
                            Jb[r][c] = jrc;
                        }
                        y[r] = e[row0 + r] - s;                                  // de_bar (pik.cpp:49)
                        for (int k = 0; k < nb; ++k) {                           // Jbar = J_i P (pik.cpp:51)
                            T t = T(0);
                            for (int c = 0; c < nv; ++c) t += J[row0 + r][c] * Wall[k][c];
                            for (int c = 0; c < nv; ++c) Jb[r][c] -= t * Wall[k][c];
                        }
                    }
                    // (Jb Jb^T + lambda^2 I) z = de, LDL^T, packed lower triangle
                    for (int i = 0; i < mi; ++i)
                        for (int j = 0; j <= i; ++j) {
                            T s = T(0);
                            for (int c = 0; c < nv; ++c) s += Jb[i][c] * Jb[j][c];
                            G[i * (i + 1) / 2 + j] = s + (i == j ? a.pik_lambda2[lvl] : T(0));
                        }
                    for (int j = 0; j < mi; ++j) {
                        T d = G[j * (j + 1) / 2 + j];
                        for (int k = 0; k < j; ++k) {
                            const T l = G[j * (j + 1) / 2 + k];
                            d -= l * l * G[k * (k + 1) / 2 + k];
                        }
                        G[j * (j + 1) / 2 + j] = d;
                        const T inv = rcp_(d);
                        for (int i = j + 1; i < mi; ++i) {
                            T s = G[i * (i + 1) / 2 + j];
                            for (int k = 0; k < j; ++k) s -= G[i * (i + 1) / 2 + k] * G[j * (j + 1) / 2 + k] * G[k * (k + 1) / 2 + k];
                            G[i * (i + 1) / 2 + j] = s * inv;
                        }
                    }
                    for (int i = 0; i < mi; ++i) {
                        T s = y[i];
                        for (int k = 0; k < i; ++k) s -= G[i * (i + 1) / 2 + k] * y[k];
                        y[i] = s;
                    }
                    for (int i = 0; i < mi; ++i) y[i] *= rcp_(G[i * (i + 1) / 2 + i]);
                    for (int i = mi - 1; i >= 0; --i) {
                        T s = y[i];
                        for (int k = i + 1; k < mi; ++k) s -= G[k * (k + 1) / 2 + i] * y[k];
                        y[i] = s;
                    }
                    for (int c = 0; c < nv; ++c) {                              // dq -= Jb^T z (pik.cpp:54-55)
                        T s = T(0);
                        for (int i = 0; i < mi; ++i) s += Jb[i][c] * y[i];
                        dq[c] -= s;
                    }
                    // projector update (pik.cpp:58-61): append this level's row-space basis
                    if (lvl != last_lvl) nb += rowspace_basis<T, NV, M>(Jb, mi, nv, Wall + nb, y);
                    row0 += mi;
                }
                // dq += P da with da = 0 (pik.cpp:65, pik.hpp:39)
            } else {
                // ---- Gram matrix + damping (dls.cpp:39-41), packed lower triangle.  Only the columns both rows can touch
                //      (the bounding range of P.row_cols[i] & P.row_cols[j], known at finalize) enter a dot product, in
                //      ascending order -- the skipped terms are exact zeros, so the sums equal the dense ones. ----
                for (int i = 0; i < rows; ++i) {
                    T *Gi = G + i * (i + 1) / 2;
                    const uint64_t mi = P.row_cols[i];
                    for (int j = 0; j <= i; ++j) {
                        T s = T(0);
                        const uint64_t mm = mi & P.row_cols[j];
                        if (mm) {  // the bounding range of the common columns: a plain loop the compiler can pipeline
                            const int c1 = 64 - __clzll((long long)mm);
                            for (int c = __ffsll((long long)mm) - 1; c < c1; ++c) s += J[i][c] * J[j][c];
                        }
                        Gi[j] = s + (i == j ? a.damping2 : T(0));
                    }
                }
                // ---- LDL^T (G is SPD thanks to the damping, so no pivoting is needed; SURVEY 8a notes); column j:
                //      v_k = L_jk D_k once, then one FMA per term ----
                for (int j = 0; j < rows; ++j) {
                    T *Gj = G + j * (j + 1) / 2;
                    T d = Gj[j];
                    for (int k = 0; k < j; ++k) {
                        const T v = Gj[k] * G[k * (k + 1) / 2 + k];
                        y[k] = v;
                        d -= Gj[k] * v;
                    }
                    Gj[j] = d;
                    const T inv = rcp_(d);
                    for (int i = j + 1; i < rows; ++i) {
                        T *Gi = G + i * (i + 1) / 2;
                        T s = Gi[j];
                        for (int k = 0; k < j; ++k) s -= Gi[k] * y[k];
                        Gi[j] = s * inv;
                    }
                }
                for (int i = 0; i < rows; ++i) {
                    const T *Gi = G + i * (i + 1) / 2;
                    T s = e[i];
                    for (int k = 0; k < i; ++k) s -= Gi[k] * y[k];
                    y[i] = s;
                }
                for (int i = 0; i < rows; ++i) y[i] *= rcp_(G[i * (i + 1) / 2 + i]);
                for (int i = rows - 1; i >= 0; --i) {
                    T s = y[i];
                    for (int k = i + 1; k < rows; ++k) s -= G[k * (k + 1) / 2 + i] * y[k];
                    y[i] = s;
                }
                // ---- dq = -J^T y (dls.cpp:52), rows that can touch column c only ----
                for (int c = 0; c < nv; ++c) {
                    T s = T(0);
                    const uint64_t mm = P.col_rows[c];
                    if (mm) {
                        const int i1 = 64 - __clzll((long long)mm);
                        for (int i = __ffsll((long long)mm) - 1; i < i1; ++i) s += J[i][c] * y[i];
                    }
                    dq[c] = -s;
                }
                // ---- FrameConstraints (dls.cpp:26-34,44-52): dq <- (I - Jc^+ Jc) dq ----
                if (P.nconstraints > 0) {
                    T Jc[kMaxConstraintRows][NV], Wc[kMaxConstraintRows][NV], dscr[kMaxConstraintRows];
                    for (int r = 0; r < P.crows; ++r)
                        for (int c = 0; c < nv; ++c) Jc[r][c] = T(0);
                    int crow = 0;
                    for (int k = 0; k < P.nconstraints; ++k) {
                        const int f = P.c_frame[k], r = P.c_ref[k], fj = P.f_parent[f], rj = P.f_parent[r];
                        const int full = P.c_type[k] == IKB_FULL, r0 = P.c_type[k] == IKB_ORIENTATION ? 3 : 0, dim = full ? 6 : 3;
                        T Rf[9], pf[3], Rr[9], pr[3], Rm[9], pm[3];
                        se3_mul(oR[fj], op[fj], P.f_placement[f], P.f_placement[f] + 9, Rf, pf);
                        se3_mul(oR[rj], op[rj], P.f_placement[r], P.f_placement[r] + 9, Rr, pr);
                        se3_actinv(Rr, pr, Rf, pf, Rm, pm);  // rMf (frame.hpp:407)
                        // + frame Jacobian, LOCAL (frame.hpp:410-411)
                        for (int j = fj; j > 0; j = P.parent[j]) {
                            const int ncol = P.jtype[j] == IKB_J_FREEFLYER ? 6 : 1;
                            for (int cc = 0; cc < ncol; ++cc) {
                                T v[3], ww[3], pxw[3], d[3], col[6];
                                world_column<T, NJ>(P, j, cc, oR, op, v, ww);
                                cross3(pf, ww, pxw);
                                d[0] = v[0] - pxw[0]; d[1] = v[1] - pxw[1]; d[2] = v[2] - pxw[2];
                                rotT_vec(Rf, d, col);
                                rotT_vec(Rf, ww, col + 3);
                                for (int i = 0; i < dim; ++i) Jc[crow + i][P.idx_v[j] + cc] += col[r0 + i];
                            }
                        }
                        // - rMf.toActionMatrixInverse() * reference frame Jacobian, LOCAL (frame.hpp:414-436)
                        for (int j = rj; j > 0; j = P.parent[j]) {
                            const int ncol = P.jtype[j] == IKB_J_FREEFLYER ? 6 : 1;
                            for (int cc = 0; cc < ncol; ++cc) {
                                T v[3], ww[3], pxw[3], d[3], lv[3], lw[3], col[6];
                                world_column<T, NJ>(P, j, cc, oR, op, v, ww);
                                cross3(pr, ww, pxw);
                                d[0] = v[0] - pxw[0]; d[1] = v[1] - pxw[1]; d[2] = v[2] - pxw[2];
                                rotT_vec(Rr, d, lv);
                                rotT_vec(Rr, ww, lw);
                                cross3(pm, lw, pxw);
                                d[0] = lv[0] - pxw[0]; d[1] = lv[1] - pxw[1]; d[2] = lv[2] - pxw[2];
                                rotT_vec(Rm, d, col);
                                rotT_vec(Rm, lw, col + 3);
                                for (int i = 0; i < dim; ++i) Jc[crow + i][P.idx_v[j] + cc] -= col[r0 + i];
                            }
                        }
                        crow += dim;
                    }
                    const int rank = rowspace_basis<T, NV, kMaxConstraintRows>(Jc, P.crows, nv, Wc, dscr);
                    for (int r = 0; r < rank; ++r) {
                        T s = T(0);
                        for (int c = 0; c < nv; ++c) s += Wc[r][c] * dq[c];
                        for (int c = 0; c < nv; ++c) dq[c] -= s * Wc[r][c];
                    }
                }
            }
            T res = T(0);
            for (int i = 0; i < P.rows_p0; ++i) res += e[i] * e[i];
            const bool converged = res < a.tolerance;
            bool finished = converged;
            if (!converged) {
                // ---- integrate (dls.cpp:67-68) + clamp (common.hpp:53-56) ----
                for (int j = 1; j < P.njoints; ++j) {
                    const int iq = P.idx_q[j], iv = P.idx_v[j];
                    if (P.jtype[j] == IKB_J_FREEFLYER) {
                        T v6[6], R0[9];
#pragma unroll
                        for (int i = 0; i < 6; ++i) v6[i] = a.step_length * dq[iv + i];
                        quat_to_rot(q[iq + 3], q[iq + 4], q[iq + 5], q[iq + 6], R0);
                        integrate_freeflyer(R0, &q[iq], &q[iq + 3], v6);
                    } else if (is_continuous(P.jtype[j])) {   // SpecialOrthogonalOperation<2>::integrate
                        T sw, cw;
                        sincos_(a.step_length * dq[iv], &sw, &cw);
                        const T c1 = cw * q[iq] - sw * q[iq + 1], s1 = sw * q[iq] + cw * q[iq + 1];
                        const T al = (T(3) - (c1 * c1 + s1 * s1)) / T(2);
                        q[iq] = c1 * al;
                        q[iq + 1] = s1 * al;
                    } else {
                        q[iq] += a.step_length * dq[iv];
                    }
                }
                for (int k = 0; k < nq; ++k) q[k] = min_(P.upper[k], max_(q[k], P.lower[k]));
                ++it;
                finished = it >= a.max_iterations;
            }
            if (finished) {
                for (int k = 0; k < nq; ++k) a.q[k * a.q_es + b * a.q_bs] = q[k];
                if (a.success) a.success[b] = converged ? 1 : 0;
                if (a.iters) a.iters[b] = it;
                if (a.resid) a.resid[b] = res;
                fetch();
            } else if (it >= a.it_cap) {
                // straggler: park it for the second launch
                for (int k = 0; k < nq; ++k) a.q[k * a.q_es + b * a.q_bs] = q[k];
                a.iters_ws[b] = it;
                a.list[atomicAdd(a.list_count, 1ULL)] = (unsigned int)b;
                fetch();
            }
        }
    }
}

}  // namespace ikb
