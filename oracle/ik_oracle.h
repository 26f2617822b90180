/*
 * ik_oracle.h -- CPU ORACLE (test infrastructure, NOT product code).
 *
 * Plain-C FP64 restatement of the reference's damped-least-squares IK path
 * (dazzmo/ik: ik/ik/dls.cpp:5-78, data.cpp:25-58, frame.hpp:37-62,152-182,
 * posture.hpp:50-67, common.hpp:47-56, visitor.hpp:15-21) and of the
 * Pinocchio / Eigen algorithms that path calls (neither library is vendored in
 * the reference nor installed here; see SURVEY.md 8c).
 *
 * PARITY UNPINNED: the reference's own tests hold no golden vector for this
 * path (every TEST body is commented out, ik/test/dls.cpp:10-76) and the
 * reference cannot be compiled here (needs Pinocchio, Eigen>=3.4, Boost, glog).
 * The oracle is therefore validated from first principles in tests/ (exp/log
 * round trips, finite-difference Jacobians, hand-derived FK) and against the
 * provisional known answers recorded in SURVEY.md 8c.
 *
 * Which Pinocchio is restated.  The reference pins no version (find_package(pinocchio
 * REQUIRED), ik/ik/CMakeLists.txt:3); its toolchain markers (GLOG_USE_GLOG_EXPORT,
 * task.hpp:3; Eigen::Vector<T,N>, common.hpp:23) put it in the Pinocchio 2.7 / 3.x era,
 * and the formulas below are those of that era's spatial/explog.hpp, explog-quaternion.hpp,
 * multibody/liegroup/special-euclidean.hpp and math/taylor-expansion.hpp, with these
 * switches (so that a reader who has Pinocchio can check them one by one):
 *   log3:   theta = acos((tr R - 1)/2), clamped to [0, pi] when the trace leaves [-1, 3];
 *           theta >= pi - 1e-2 -> the diagonal-based formula  w_i = sign(R_kj - R_jk) *
 *           theta * sqrt(max(0, (R_ii - cos theta) / (1 - cos theta)));  else
 *           w = (theta > precision<2>() ? theta / (2 sin theta) : 1/2) * vee(R - R^T)
 *   Taylor switches: TaylorSeriesExpansion<double>::precision<n>() = eps^(1/(n+1)):
 *           precision<3>() = 1.2207e-4 (log6 alpha/beta, Jlog3 / Jlog6 coefficients, exp3 /
 *           exp6 coefficients), precision<2>() = 6.0555e-6 (log3 scale factor)
 *   log6:   alpha = 1 - t^2/12 - t^4/720, beta = 1/12 + t^2/720 below the switch, the closed
 *           forms with sin / cos of theta above it; Jlog6 block B = C A with beta_dot =
 *           1/360 below the switch
 *   integrate (SE3): M1 = M0 exp6(v); quaternion from the rotation matrix (Eigen's branch
 *           on the trace), sign chosen so that dot(q_new, q_old) >= 0, then the first-order
 *           renormalisation q *= (3 - |q|^2)/2 (quaternion::firstOrderNormalize)
 *   LDLT:   Eigen::LDLT with its diagonal pivoting (largest |diagonal| first) and D^+ with
 *           the tolerance 1 / numeric_limits::highest (Eigen 3.4 solveInPlace)
 * Releases of Pinocchio older than 2.6 use fixed 1e-8-style switches instead of the
 * precision<n>() ones; results then differ at the 1e-12 level near theta = 1e-4 only.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
 * reference legs may load this library; the product (ik_b200/) never does.
 *
 * Conventions: SE3 = 12 doubles, rotation row-major R[0..8] then p[0..2];
 * motion vectors are [linear; angular]; free-flyer q = [p(3), quat x,y,z,w].
 */
#ifndef IK_ORACLE_H
#define IK_ORACLE_H

#ifdef __cplusplus
extern "C" {
#endif

enum { IKO_J_UNIVERSE = 0, IKO_J_FREEFLYER = 1, IKO_J_RX = 2, IKO_J_RY = 3, IKO_J_RZ = 4,
       IKO_J_REV_UNALIGNED = 5, IKO_J_PX = 6, IKO_J_PY = 7, IKO_J_PZ = 8, IKO_J_PRIS_UNALIGNED = 9 };

enum { IKO_TASK_FRAME = 0, IKO_TASK_ALIGN_AXIS = 1, IKO_TASK_POSTURE = 2, IKO_TASK_COM = 3 };
enum { IKO_POSITION = 0, IKO_ORIENTATION = 1, IKO_FULL = 2 };

typedef struct {
    int njoints; /* including the universe joint 0 */
    int nq, nv;
    const int *parent;       /* [njoints] */
    const int *jtype;        /* [njoints] */
    const int *idx_q;        /* [njoints] */
    const int *idx_v;        /* [njoints] */
    const double *placement; /* [njoints][12] joint placement in the parent joint frame */
    const double *axis;      /* [njoints][3] (unaligned joints) */
    const double *lower;     /* [nq] */
    const double *upper;     /* [nq] */
    int nframes;
    const int *frame_parent;       /* [nframes] supporting joint */
    const double *frame_placement; /* [nframes][12] */
    /* per joint: total mass of the bodies it supports and their centre of mass in the joint frame (Pinocchio
     * model.inertias[j].mass() / .lever(); CentreOfMassTask, centre_of_mass.hpp:14-52) */
    const double *mass;            /* [njoints] */
    const double *com;             /* [njoints][3] */
} iko_model;

typedef struct {
    int ntasks;
    int max_priority_level;
    const int *kind;     /* [ntasks] IKO_TASK_* */
    const int *frame;    /* [ntasks] task frame (FRAME, ALIGN_AXIS) */
    const int *ref;      /* [ntasks] reference frame */
    const int *type;     /* [ntasks] FRAME: IKO_POSITION/ORIENTATION/FULL; ALIGN_AXIS: axis 0/1/2; POSTURE: nj */
    const int *priority; /* [ntasks] */
    const double *weight; /* concatenated per-row weights, task insertion order */
    const double *mask;   /* concatenated posture masks (POSTURE tasks only, insertion order) */
    /* FrameConstraints (frame.hpp:333-465, problem.hpp add_frame_constraint): ik::dls projects its step into the null
     * space of their stacked Jacobian (dls.cpp:26-34,44-49) */
    int nconstraints;
    const int *c_frame;  /* [nconstraints] */
    const int *c_ref;    /* [nconstraints] reference frame */
    const int *c_type;   /* [nconstraints] IKO_POSITION / ORIENTATION / FULL */
} iko_problem;

typedef struct {
    int max_iterations;  /* common.hpp:61 (default 100) */
    double step_length;  /* common.hpp:65 (default 1.0) */
    double damping;      /* dls.hpp:25 (default 1e-2) */
    double tolerance;    /* visitor.hpp:19: squared-norm threshold, 1e-4 */
} iko_params;

/* sizes */
int iko_task_dim(const iko_problem *pb, int t);
int iko_task_target_size(const iko_problem *pb, int t);
int iko_target_size(const iko_problem *pb);          /* doubles per problem */
int iko_e_size(const iko_problem *pb, int priority); /* problem.hpp:34-40 */
int iko_total_rows(const iko_problem *pb);

/* Lie-group primitives (Pinocchio explog.hpp restated) */
void iko_exp3(const double w[3], double R[9]);
void iko_log3(const double R[9], double w[3], double *theta);
void iko_exp6(const double v[6], double M[12]);
void iko_log6(const double M[12], double v[6]);
void iko_Jlog3(double theta, const double w[3], double J[9]);
void iko_Jlog6(const double M[12], double J[36]);
void iko_se3_mul(const double A[12], const double B[12], double C[12]);    /* A*B */
void iko_se3_actinv(const double A[12], const double B[12], double C[12]); /* A^-1*B */
void iko_quat_to_rot(const double q_xyzw[4], double R[9]);
void iko_rot_to_quat(const double R[9], double q_xyzw[4]);

/* kinematics */
void iko_fk(const iko_model *m, const double *q, double *oMi /*[njoints][12]*/);
void iko_frame_placement(const iko_model *m, const double *oMi, int frame, double oMf[12]);
void iko_joint_jacobians(const iko_model *m, const double *oMi, double *J /*[6][nv] row-major, world*/);
void iko_frame_jacobian_local(const iko_model *m, const double *oMi, const double *Jworld, int frame,
                              double *Jf /*[6][nv]*/);
void iko_integrate(const iko_model *m, const double *q, const double *v, double *qout);
void iko_clip(const iko_model *m, double *q);

/* one evaluate_problem_data() (data.cpp:25-58): stacked e [rows] and J [rows][nv] */
void iko_evaluate(const iko_model *m, const iko_problem *pb, const double *q, const double *targets,
                  double *e, double *J);

/* pinocchio::centerOfMass / jacobianCenterOfMass (data.cpp:31-34): com [3] and Jcom [3][nv] in the world frame */
void iko_center_of_mass(const iko_model *m, const double *q, double com[3], double *Jcom);

/* rows of all FrameConstraints and their stacked Jacobian Jc [crows][nv] (FrameConstraint::compute_jacobian,
 * frame.hpp:399-437: frame Jacobian minus the reference frame's, both LOCAL, the latter moved by rMf^-1) */
int iko_c_size(const iko_problem *pb);
void iko_constraint_jacobian(const iko_model *m, const iko_problem *pb, const double *q, double *Jc);

/* Eigen LDLT (pivoted, lower, unblocked) restated: solves A x = b, A n x n row-major (destroyed) */
void iko_ldlt_solve(int n, double *A, const double *b, double *x);

/* ik::dls (dls.cpp:5-78).  Returns success (1/0).  iters = steps taken; resid = ||e[0]||^2 at the last
 * evaluation; dq_out (optional, nv) = last step direction. */
int iko_dls(const iko_model *m, const iko_problem *pb, const iko_params *prm, const double *q0,
            const double *targets, double *q_out, int *iters, double *resid, double *dq_out);

/* Loop of iko_dls over a batch, AoS: q0 [B][nq], targets [B][tsz]; nthreads >= 1 (pthreads). */
void iko_dls_batch(const iko_model *m, const iko_problem *pb, const iko_params *prm, int B,
                   const double *q0, const double *targets, double *q_out, unsigned char *success,
                   int *iters, double *resid, int nthreads);

/* ---- ik::pik, priority-based IK (pik.cpp:5-96, pik.hpp:13-57) ---- */
#define IKO_MAX_LEVELS 8
typedef struct {
    int max_iterations;              /* pik.hpp:14 (default 100) */
    double step_length;              /* pik.hpp:16 (default 1.0) */
    double tolerance;                /* visitor.hpp:19 */
    double lambda[IKO_MAX_LEVELS];   /* pik_data::lambda, damping per priority level (pik.hpp:31: 1.0) */
} iko_pik_params;
/* damp_pseudoinverse(M, lambda) (pik.cpp:5-21): M m x n row-major (m <= n) -> out n x m */
void iko_damp_pseudoinverse(int m, int n, const double *M, double lambda, double *out);
/* M.completeOrthogonalDecomposition().pseudoInverse() * M (pik.cpp:59-61) -> proj n x n; returns the numerical rank */
int iko_rowspace_projector(int m, int n, const double *M, double *proj);
/* ik::pik on one problem / a batch.  Both return -1 and touch no output when a task's priority has no lambda (at or
 * above IKO_MAX_LEVELS); otherwise iko_pik returns success (1/0) and iko_pik_batch 0. */
int iko_pik(const iko_model *m, const iko_problem *pb, const iko_pik_params *prm, const double *q0,
            const double *targets, double *q_out, int *iters, double *resid, double *dq_out);
int iko_pik_batch(const iko_model *m, const iko_problem *pb, const iko_pik_params *prm, int B, const double *q0,
                  const double *targets, double *q_out, unsigned char *success, int *iters, double *resid,
                  int nthreads);

#ifdef __cplusplus
}
#endif
#endif
