// Host-only: fills the device constant blob (dev_problem.hpp) of a finalized problem -- model constants, tasks in stacked
// order, Jacobian sparsity masks and the index tables of the team-per-problem kernel (dls_coop.cuh).  Shared by
// ikb_problem_finalize (ikb_capi.cu) and the g++-built unit-test harness (tests/cpu_harness/coop_harness.cpp), so the
// tables the CPU tests exercise are the ones the GPU kernel reads.
#pragma once
#include <algorithm>
#include <cstring>
#include <limits>
#include <vector>

#include "dev_problem.hpp"
#include "model.hpp"

namespace ikb {

// stacked order: priority level, then insertion order (dls.cpp:18-24)
inline std::vector<int> stacked_order(const HostProblem &hp) {
    std::vector<int> order(hp.tasks.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return hp.tasks[a].priority < hp.tasks[b].priority; });
    return order;
}

// model frames referenced by tasks / constraints (task frame, reference frame), in first-use order
inline std::vector<int> used_frames(const HostProblem &hp) {
    std::vector<int> used;
    for (const auto &t : hp.tasks)
        if (t.kind != IKB_TASK_POSTURE)
            for (int f : {t.kind == IKB_TASK_COM ? t.ref : t.frame, t.ref})
                if (std::find(used.begin(), used.end(), f) == used.end()) used.push_back(f);
    for (const auto &c : hp.constraints)
        for (int f : {c.frame, c.ref})
            if (std::find(used.begin(), used.end(), f) == used.end()) used.push_back(f);
    if (used.empty()) used.push_back(0);
    return used;
}

// Index tables of dls_coop.cuh: which joints need a world placement, the root-to-leaf paths that cover them, and the
// (task, joint, velocity coordinate) triples whose Jacobian entries are structurally non-zero.  False when the problem
// exceeds the table capacities (the caller then keeps the thread-per-problem fallback).
inline bool build_coop_tables(const HostProblem &hp, const std::vector<int> &order, CoopTables &C) {
    const HostModel &m = hp.model;
    std::memset(&C, 0, sizeof(C));
    {
        const std::vector<int> used = used_frames(hp);
        const SE3d id = se3_identity();
        for (size_t f = 0; f < used.size() && f < (size_t)kMaxFrames; ++f) {
            bool is_id = true;
            for (int k = 0; k < 12; ++k) is_id = is_id && m.frame_placement[used[f]][k] == id[k];
            C.f_ident[f] = is_id ? (m.frame_parent[used[f]] == 0 ? 2 : 1) : 0;
        }
    }
    const int nj = m.njoints();
    std::vector<char> need(nj, 0);
    auto mark = [&](int frame) {
        for (int j = m.frame_parent[frame]; j > 0; j = m.parent[j]) need[j] = 1;
    };
    for (const auto &t : hp.tasks) {
        if (t.kind == IKB_TASK_POSTURE) continue;
        if (t.kind == IKB_TASK_COM) {
            C.has_com = 1;
            for (int j = 1; j < nj; ++j) need[j] = 1;
        } else {
            mark(t.frame);
        }
        mark(t.ref);
    }
    for (const auto &c : hp.constraints) {
        mark(c.frame);
        mark(c.ref);
    }
    std::vector<char> has_child(nj, 0);
    for (int j = 1; j < nj; ++j)
        if (need[j] && m.parent[j] > 0) has_child[m.parent[j]] = 1;
    for (int j = 1; j < nj; ++j) {
        if (!need[j]) continue;
        C.fkj[C.n_fkj++] = (uint8_t)j;
        if (has_child[j]) continue;
        if (C.npaths >= kCoopMaxPaths) return false;
        std::vector<int> chain;
        for (int k = j; k > 0; k = m.parent[k]) chain.push_back(k);
        std::reverse(chain.begin(), chain.end());
        C.path_len[C.npaths] = (uint8_t)chain.size();
        for (size_t k = 0; k < chain.size(); ++k) C.path_joint[C.npaths][k] = (uint8_t)chain[k];
        ++C.npaths;
    }
    for (size_t s = 0; s < order.size(); ++s) {
        const HostTask &t = hp.tasks[order[s]];
        if (t.kind == IKB_TASK_POSTURE) continue;
        std::vector<int> joints;
        if (t.kind == IKB_TASK_COM)
            for (int j = 1; j < nj; ++j) joints.push_back(j);
        else
            for (int j = m.frame_parent[t.frame]; j > 0; j = m.parent[j]) joints.push_back(j);
        for (int j : joints)
            for (int cc = 0; cc < joint_nv(m.jtype[j]); ++cc) {
                if (C.npairs >= kCoopMaxPairs) return false;
                C.pair_task[C.npairs] = (uint8_t)s;
                C.pair_joint[C.npairs] = (uint8_t)j;
                C.pair_cc[C.npairs] = (uint8_t)cc;
                ++C.npairs;
            }
    }
    return true;
}

template <typename T>
inline void fill_dev_problem(const HostProblem &hp, const std::vector<int> &order, const std::vector<int> &used_frames,
                      DevProblem<T> &P) {
    const HostModel &m = hp.model;
    std::memset(&P, 0, sizeof(P));
    P.njoints = m.njoints();
    P.nq = m.nq;
    P.nv = m.nv;
    P.nframes = (int)used_frames.size();
    P.ntasks = (int)hp.tasks.size();
    P.rows = hp.rows();
    P.rows_p0 = hp.e_size(0);
    P.nconstraints = (int)hp.constraints.size();
    P.crows = hp.c_size();
    for (size_t k = 0; k < hp.constraints.size(); ++k) {
        auto lf = [&](int fid) { return (int)(std::find(used_frames.begin(), used_frames.end(), fid) - used_frames.begin()); };
        P.c_frame[k] = lf(hp.constraints[k].frame);
        P.c_ref[k] = lf(hp.constraints[k].ref);
        P.c_type[k] = hp.constraints[k].type;
    }
    P.nlevels = hp.levels();
    for (int l = 0; l < kPikMaxLevels; ++l) P.level_rows[l] = l < P.nlevels ? hp.e_size(l) : 0;
    P.tsz = hp.target_size();
    for (int j = 0; j < m.njoints(); ++j) {
        P.parent[j] = m.parent[j];
        P.jtype[j] = m.jtype[j];
        P.idx_q[j] = m.idx_q[j];
        P.idx_v[j] = m.idx_v[j];
        for (int k = 0; k < 12; ++k) P.placement[j][k] = (T)m.placement[j][k];
        for (int k = 0; k < 3; ++k) P.axis[j][k] = (T)m.axis[j][k];
    }
    double tm = 0;
    for (int j = 0; j < m.njoints(); ++j) {
        P.mass[j] = (T)m.mass[j];
        for (int k = 0; k < 3; ++k) P.com[j][k] = (T)m.com[j][k];
        if (j >= 1) tm += m.mass[j];
    }
    P.total_mass = (T)tm;
    const double big = (double)std::numeric_limits<T>::max();
    for (int k = 0; k < m.nq; ++k) {
        P.lower[k] = (T)std::max(m.lower[k], -big);
        P.upper[k] = (T)std::min(m.upper[k], big);
    }
    for (size_t f = 0; f < used_frames.size(); ++f) {
        P.f_parent[f] = m.frame_parent[used_frames[f]];
        for (int k = 0; k < 12; ++k) P.f_placement[f][k] = (T)m.frame_placement[used_frames[f]][k];
    }
    auto local_frame = [&](int fid) {
        return (int)(std::find(used_frames.begin(), used_frames.end(), fid) - used_frames.begin());
    };
    for (auto &x : P.row_cols) x = 0;
    for (auto &x : P.col_rows) x = 0;
    int row = 0, moff = 0;
    for (size_t s = 0; s < order.size(); ++s) {
        const HostTask &t = hp.tasks[order[s]];
        // columns this task's Jacobian rows can touch
        uint64_t cols = 0;
        if (t.kind == IKB_TASK_POSTURE) {
            for (int i = 0; i < t.type; ++i) cols |= 1ULL << (m.nv - t.type + i);
        } else if (t.kind == IKB_TASK_COM) {
            cols = m.nv >= 64 ? ~0ULL : ((1ULL << m.nv) - 1);
        } else {
            for (int j = m.frame_parent[t.frame]; j > 0; j = m.parent[j])
                for (int k = 0; k < joint_nv(m.jtype[j]); ++k) cols |= 1ULL << (m.idx_v[j] + k);
        }
        for (int i = 0; i < t.dim; ++i) {
            P.row_cols[row + i] = cols;
            for (int c = 0; c < m.nv; ++c)
                if (cols >> c & 1) P.col_rows[c] |= 1ULL << (row + i);
        }
        P.t_kind[s] = t.kind;
        P.t_frame[s] = (t.kind == IKB_TASK_POSTURE || t.kind == IKB_TASK_COM) ? 0 : local_frame(t.frame);
        P.t_ref[s] = t.kind == IKB_TASK_POSTURE ? 0 : local_frame(t.ref);
        P.t_type[s] = t.type;
        P.t_row[s] = row;
        P.t_dim[s] = t.dim;
        P.t_toff[s] = hp.target_offset(order[s]);
        P.t_moff[s] = moff;
        for (int i = 0; i < t.dim; ++i) P.weight[row + i] = (T)t.weight[i];
        if (t.kind == IKB_TASK_POSTURE) {
            for (int i = 0; i < t.type; ++i) P.mask[moff + i] = (T)t.mask[i];
            moff += t.type;
        }
        row += t.dim;
    }
    P.coop_ok = build_coop_tables(hp, order, P.coop) ? 1 : 0;
}

}  // namespace ikb
