// Device-side constant blob of one IK problem (model + tasks), one instance per scalar type.
//
// This is the "URDF constants" block of the design: ~10 KB, read-only, identical for every problem of a
// batch.  It is written once into HBM by ikb_problem_finalize() and every CTA stages it into shared memory
// with one TMA bulk copy (cp.async.bulk) at kernel start; lanes then read it through shared-memory
// broadcasts.  Tasks are stored in STACKED order (priority level, then insertion order; reference
// dls.cpp:18-24) so the kernel never sorts.
#pragma once
#include <cstdint>

namespace ikb {

constexpr int kMaxJoints = 48;
constexpr int kMaxNq = 64;
constexpr int kMaxTasks = 16;
constexpr int kMaxFrames = 32;  // frames referenced by tasks (task frames + reference frames)
constexpr int kMaxRows = 48;
constexpr int kMaxConstraints = 4;   // FrameConstraints
constexpr int kMaxConstraintRows = 12;
constexpr int kPikMaxLevels = 7;     // priority levels ik::pik walks (level_rows, pik_lambda2, ikb_pik_params::lambda)

// Index tables of the team-per-problem kernel (dls_coop.cuh), built by build_coop_tables (problem_fill.hpp).
constexpr int kCoopMaxPaths = 16;
constexpr int kCoopMaxPairs = 192;
struct alignas(16) CoopTables {
    int32_t n_fkj;    // joints whose world placement some task / constraint needs (all joints with a CentreOfMassTask)
    int32_t npaths;   // root-to-leaf paths covering them
    int32_t npairs;   // structurally non-zero (task, joint, velocity coordinate) triples of the stacked Jacobian
    int32_t has_com;
    uint8_t fkj[kMaxJoints];
    uint8_t path_len[kCoopMaxPaths];
    uint8_t path_joint[kCoopMaxPaths][kMaxJoints];
    uint8_t pair_task[kCoopMaxPairs], pair_joint[kCoopMaxPairs], pair_cc[kCoopMaxPairs];
    // used frame f (index into f_parent / f_placement): 1 = its placement on the supporting joint is the identity (the
    // joint's own frame, `universe`), so oMf = oMi[parent] needs no product; 2 = it is `universe` itself (oMf = identity)
    uint8_t f_ident[kMaxFrames];
};

template <typename T> struct alignas(16) DevProblem {
    int32_t njoints, nq, nv, nframes, ntasks, rows, rows_p0, tsz;
    int32_t parent[kMaxJoints], jtype[kMaxJoints], idx_q[kMaxJoints], idx_v[kMaxJoints];
    T placement[kMaxJoints][12];
    T axis[kMaxJoints][3];
    T lower[kMaxNq], upper[kMaxNq];
    T mass[kMaxJoints];        // per joint: mass of the bodies it supports, their centre of mass in the joint frame
    T com[kMaxJoints][3];      //   (CentreOfMassTask, centre_of_mass.hpp:14-52); total_mass = sum over joints >= 1
    T total_mass, tm_pad_;
    int32_t f_parent[kMaxFrames];
    T f_placement[kMaxFrames][12];
    // tasks, stacked order
    int32_t t_kind[kMaxTasks], t_frame[kMaxTasks], t_ref[kMaxTasks], t_type[kMaxTasks];
    int32_t t_row[kMaxTasks], t_dim[kMaxTasks], t_toff[kMaxTasks], t_moff[kMaxTasks];
    T weight[kMaxRows];  // stacked row order
    T mask[kMaxNq];      // posture masks, concatenated in stacked order
    // FrameConstraints (frame.hpp:333-465): frame / reference frame (indices into f_parent / f_placement) and KinematicType
    int32_t nconstraints, crows;
    int32_t c_frame[kMaxConstraints], c_ref[kMaxConstraints], c_type[kMaxConstraints], c_pad_[2];
    // priority levels up to the highest one a task uses (not max_priority_level + 1: empty top levels cost nothing and
    // may exceed the table).  ik::pik walks level_rows[0 .. nlevels); its entry points refuse nlevels > kPikMaxLevels,
    // ik::dls never reads either field.
    int32_t nlevels;
    int32_t level_rows[kPikMaxLevels];   // rows of priority level l (stacked order = level by level)
    int32_t pad_[4];           // keeps sizeof a multiple of 16 for the bulk copy
    // Sparsity of the stacked task Jacobian, known when the problem is finalized (a frame task only touches the columns of
    // the joints between the root and its frame; SURVEY 8a: the reference's dense products ignore 60 % zeros): bit c of
    // row_cols[r] = column c of row r may be non-zero, bit r of col_rows[c] likewise (supersets; nv, rows <= 64).
    uint64_t row_cols[kMaxRows];
    uint64_t col_rows[kMaxNq];
    CoopTables coop;
    int32_t coop_ok, coop_pad_[3];
};

constexpr int kMaxSegments = 8;

// One batch of a MERGED launch (pipelined queue, ikb_queue_*): problems [begin, begin + its B) of the launch live in
// these buffers (same meaning as the fields of SolveArgs / ikb_batch_io).
template <typename T> struct BatchSeg {
    const T *q0; long long q0_es, q0_bs;
    const T *targets; long long tg_es, tg_bs;
    T *q; long long q_es, q_bs;
    unsigned char *success;
    int *iters;
    T *resid;
    long long begin;
};

// Per-launch arguments (passed by value as a kernel parameter).
template <typename T> struct SolveArgs {
    const T *q0; long long q0_es, q0_bs;
    const T *targets; long long tg_es, tg_bs;
    T *q; long long q_es, q_bs;
    unsigned char *success;
    int *iters;
    T *resid;
    unsigned long long *ticket;  // work-stealing counter, zeroed before the launch
    long long B;
    int max_iterations;
    T step_length, damping2, tolerance;
    // Two-phase scheduling of the specialised kernels (dls_spec.cuh): the BULK launch suspends a problem that has not
    // finished after `it_cap` steps (its iterate goes to `q`, its step count to `iters_ws`, its index to `list`); the
    // TAIL launch (`resume` = 1) takes its problems from `list` and continues them from `q` / `iters_ws`.
    int it_cap;                       // >= max_iterations: never suspend
    int resume;                       // 0: tickets are problem indices 0..B-1; 1: tickets index `list`
    unsigned int *list;               // suspended problem indices
    unsigned long long *list_count;   // number of entries in `list` (zeroed before the BULK launch)
    int *iters_ws;                    // step counts of suspended problems (the caller's `iters` or scratch)
    // ik::pik (generic kernel only): squared damping of every priority level (pik_data::lambda, pik.hpp:31)
    T pik_lambda2[kPikMaxLevels];
    // ikb_dls_solve_ex / ikb_pik_solve_ex (team-per-problem kernel only): dls_data::dq [B][nv], stacked e [B][rows] and
    // J [B][rows][nv] of the last evaluation (data.hpp:15-28); NULL = not wanted
    T *aux_dq, *aux_e, *aux_J;
    // Merged launch: `nseg` > 0 batches, sorted by `begin`, B = their total size; q0 ... resid above are then unused and
    // iters_ws / list are indexed by the launch-wide problem index.  Unused entries have begin = LLONG_MAX.  The table
    // travels in the kernel parameters: the lookup is a handful of constant-bank compares, no memory traffic.
    int nseg;
    // dls_spec.cuh: 0 = every group of the CTA loops on its own (phases of different groups interleave on the schedulers:
    // measured +3 % on the Cassie bulk launch), 1 = the CTA's groups start every trip together (IKB_LOOP_SYNC=cta)
    int loop_sync;
    BatchSeg<T> seg[kMaxSegments];
    // Carried stragglers (pipelined queue, ikb_queue.cu): the problems the PREVIOUS merged launch suspended when its
    // ticket queue ran dry are not given a TAIL launch of their own; this launch continues them first -- tickets
    // [0, *carry_count) -- beside its own fresh problems, from the iterates / step counts the previous launch saved.  They
    // live in the previous launch's buffers (`cseg`) and are never suspended again.  carry_list == NULL: nothing carried.
    const unsigned int *carry_list;
    const unsigned long long *carry_count;
    const int *carry_iters;
    BatchSeg<T> cseg[kMaxSegments];
};

// Buffers of ONE problem, resolved from its launch-wide index (all pointers already point at the problem).
template <typename T> struct ProblemIO {
    const T *q0; long long q0_es;
    const T *targets; long long tg_es;
    T *q; long long q_es;
    unsigned char *success;
    int *iters;
    T *resid;
};
#if defined(__CUDACC__)
template <typename T> __device__ __forceinline__ ProblemIO<T> segment_io(const BatchSeg<T> (&seg)[kMaxSegments], long long b) {
    int s = 0;
#pragma unroll
    for (int i = 1; i < kMaxSegments; ++i) s += b >= seg[i].begin ? 1 : 0;
    const BatchSeg<T> &g = seg[s];
    const long long l = b - g.begin;
    return {g.q0 + l * g.q0_bs, g.q0_es, g.targets + l * g.tg_bs, g.tg_es, g.q + l * g.q_bs, g.q_es,
            g.success ? g.success + l : nullptr, g.iters ? g.iters + l : nullptr, g.resid ? g.resid + l : nullptr};
}
// SEG = false: one batch, plain pointer arithmetic on the launch arguments.
// SEG = true : merged launch, segment lookup in the (constant-bank) kernel parameters.
template <bool SEG, typename T> __device__ __forceinline__ ProblemIO<T> problem_io(const SolveArgs<T> &a, long long b) {
    if constexpr (SEG) {
        int s = 0;
#pragma unroll
        for (int i = 1; i < kMaxSegments; ++i) s += b >= a.seg[i].begin ? 1 : 0;
        const BatchSeg<T> &g = a.seg[s];
        const long long l = b - g.begin;
        return {g.q0 + l * g.q0_bs, g.q0_es, g.targets + l * g.tg_bs, g.tg_es, g.q + l * g.q_bs, g.q_es,
                g.success ? g.success + l : nullptr, g.iters ? g.iters + l : nullptr, g.resid ? g.resid + l : nullptr};
    } else {
        return {a.q0 + b * a.q0_bs, a.q0_es, a.targets + b * a.tg_bs, a.tg_es, a.q + b * a.q_bs, a.q_es,
                a.success ? a.success + b : nullptr, a.iters ? a.iters + b : nullptr, a.resid ? a.resid + b : nullptr};
    }
}
#endif

}  // namespace ikb
