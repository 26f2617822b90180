/*
 * ikb200.h -- C ABI of the B200-native batched inverse-kinematics engine (libikb200.so).
 *
 * This is the drop-in boundary for the damped-least-squares IK path of dazzmo/ik ("Puppeteer").  The
 * reference has no FFI of its own: its boundary is the C++ API in namespace ik (target ik::ik,
 * ik/ik/CMakeLists.txt:37).  Each entry point below names the reference interface it replaces; the C++
 * facade in include/ik/ re-creates the reference's class names on top of these calls and
 * INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Rules of the ABI: plain pointers and sizes only; opaque handles; every call returns an ikb_status (or a
 * non-negative index / size where documented; negative values are -ikb_status); no exceptions cross the
 * boundary; ikb_last_error() returns a thread-local message for the last failing call.  A model / problem
 * handle is immutable once ikb_problem_finalize() has run, so concurrent solves on different CUDA streams
 * are safe.  There is NO CPU fallback: solve entry points fail with IKB_ERR_CUDA / IKB_ERR_NO_DEVICE when
 * no B200-class device is usable.
 *
 * Conventions (same as Pinocchio's, which the reference inherits): SE3 = 12 scalars, rotation row-major
 * R[0..8] then translation p[0..2]; spatial vectors are [linear; angular]; a free-flyer root uses
 * q = [x y z, qx qy qz qw] (reference ik_ros/src/cassie.cpp:68-70) and a LOCAL-frame 6-vector tangent.
 */
#ifndef IKB200_H
#define IKB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IKB_VERSION 200 /* 0.2.0 */

typedef enum {
    IKB_OK = 0,
    IKB_ERR_INVALID_ARG = 1,
    IKB_ERR_PARSE = 2,         /* malformed URDF */
    IKB_ERR_UNKNOWN_FRAME = 3, /* the reference silently indexes out of range here (problem.hpp:85-92) */
    IKB_ERR_UNSUPPORTED = 4,   /* joint type / size outside what the kernels handle */
    IKB_ERR_CUDA = 5,
    IKB_ERR_NO_DEVICE = 6,
    IKB_ERR_NOT_FINALIZED = 7
} ikb_status;

/* joint types of the flattened tree (Pinocchio JointModel* equivalents).  RUB* are URDF `continuous` joints
 * (JointModelRevoluteUnbounded{X,Y,Z} / ...Unaligned): two configuration entries (cos theta, sin theta) and one velocity
 * coordinate; every other movable joint has one of each except the free-flyer (7 / 6). */
typedef enum {
    IKB_J_UNIVERSE = 0, IKB_J_FREEFLYER = 1, IKB_J_RX = 2, IKB_J_RY = 3, IKB_J_RZ = 4, IKB_J_REV_UNALIGNED = 5,
    IKB_J_PX = 6, IKB_J_PY = 7, IKB_J_PZ = 8, IKB_J_PRIS_UNALIGNED = 9,
    IKB_J_RUBX = 10, IKB_J_RUBY = 11, IKB_J_RUBZ = 12, IKB_J_RUB_UNALIGNED = 13
} ikb_joint_type;

/* ik::KinematicType, reference ik/ik/frame.hpp:20 */
typedef enum { IKB_POSITION = 0, IKB_ORIENTATION = 1, IKB_FULL = 2 } ikb_kinematic_type;
/* ik::AlignAxisType, reference ik/ik/frame.hpp:202 */
typedef enum { IKB_AXIS_X = 0, IKB_AXIS_Y = 1, IKB_AXIS_Z = 2 } ikb_axis;
typedef enum { IKB_TASK_FRAME = 0, IKB_TASK_ALIGN_AXIS = 1, IKB_TASK_POSTURE = 2, IKB_TASK_COM = 3 } ikb_task_kind;
typedef enum { IKB_F64 = 0, IKB_F32 = 1 } ikb_dtype;

typedef struct ikb_model ikb_model;     /* replaces ik::model_t = pinocchio::Model (common.hpp:17) */
typedef struct ikb_problem ikb_problem; /* replaces ik::InverseKinematicsProblem (problem.hpp:9-206) */

/* ik::dls_parameters : default_solver_parameters (dls.hpp:24-28, common.hpp:59-66).  max_time and
 * random_restart are carried for layout compatibility; the reference never reads them either. */
typedef struct {
    int32_t max_iterations; /* 100 */
    int32_t random_restart; /* 0, unused */
    double max_time;        /* 1.0, unused */
    double step_length;     /* 1.0 */
    double damping;         /* 1e-2 */
    double tolerance;       /* squared-norm stop threshold of inverse_kinematics_visitor::should_stop, 1e-4 (visitor.hpp:19) */
} ikb_dls_params;

void ikb_dls_params_default(ikb_dls_params *p);

/* Flat description of a kinematic tree, for callers that already own a parsed model. */
typedef struct {
    int32_t njoints; /* including universe joint 0 */
    const int32_t *parent;   /* [njoints] */
    const int32_t *jtype;    /* [njoints] ikb_joint_type */
    const double *placement; /* [njoints][12] */
    const double *axis;      /* [njoints][3], unaligned joints only (may be NULL otherwise) */
    const double *lower;     /* [nq] */
    const double *upper;     /* [nq] */
    const char *const *joint_names; /* [njoints] or NULL */
    int32_t nframes;
    const int32_t *frame_parent;     /* [nframes] supporting joint */
    const double *frame_placement;   /* [nframes][12] */
    const char *const *frame_names;  /* [nframes] */
} ikb_model_desc;

/* ---- model (host only) ------------------------------------------------------------------------- */
/* pinocchio::urdf::buildModelFromXML(xml, JointModelFreeFlyer(), model), reference ik_ros/src/cassie.cpp:34-35.
 * free_flyer = 0 builds the fixed-base model (buildModelFromXML(xml, model)). */
int ikb_model_from_urdf(const char *xml, size_t len, int free_flyer, ikb_model **out);
int ikb_model_from_desc(const ikb_model_desc *desc, ikb_model **out);
void ikb_model_free(ikb_model *m);
int ikb_model_njoints(const ikb_model *m);
int ikb_model_nq(const ikb_model *m); /* model.nq */
int ikb_model_nv(const ikb_model *m); /* model.nv */
int ikb_model_nframes(const ikb_model *m);
/* model.getFrameId(name) (reference common.hpp:50): index of the first frame with that name, nframes if absent */
int ikb_model_frame_id(const ikb_model *m, const char *name);
const char *ikb_model_joint_name(const ikb_model *m, int joint);
const char *ikb_model_frame_name(const ikb_model *m, int frame);
int ikb_model_get_topology(const ikb_model *m, int32_t *parent, int32_t *jtype, int32_t *idx_q, int32_t *idx_v);
int ikb_model_get_placements(const ikb_model *m, double *placement /*[njoints][12]*/, double *axis /*[njoints][3]*/);
/* model.lowerPositionLimit / upperPositionLimit (reference common.hpp:54-55) */
int ikb_model_get_limits(const ikb_model *m, double *lower, double *upper);
int ikb_model_set_limits(ikb_model *m, const double *lower, const double *upper);
int ikb_model_get_frames(const ikb_model *m, int32_t *parent_joint, int32_t *type, double *placement /*[nframes][12]*/);
int ikb_model_neutral(const ikb_model *m, double *q); /* pinocchio::neutral: zeros, unit quaternion, (1, 0) for continuous joints */

/* ---- problem (host only until finalize) --------------------------------------------------------- */
/* InverseKinematicsProblem(model, max_priority_level), reference problem.hpp:17-22 (copies the model) */
int ikb_problem_create(const ikb_model *m, int max_priority_level, ikb_problem **out);
void ikb_problem_free(ikb_problem *p);
/* FrameTask(model, frame, type, reference_frame) + add_frame_task(name, task, priority): frame.hpp:89-111,
 * problem.hpp:55-66.  weights: `dim` per-row weights (Task::weighting(), task.hpp:40) or NULL for ones.
 * Returns the task index (>= 0) or -ikb_status. */
int ikb_problem_add_frame_task(ikb_problem *p, int frame, int kinematic_type, int reference_frame, int priority,
                               const double *weights);
/* AlignAxisTask + add_align_axis_task: frame.hpp:210-319, problem.hpp:94-105 */
int ikb_problem_add_align_axis_task(ikb_problem *p, int frame, int axis, int reference_frame, int priority,
                                    const double *weights);
/* PostureTask(model, nj) + add_posture_task: posture.hpp:17-86, problem.hpp:134-145.  mask: nj entries or NULL.
 * IKB_ERR_UNSUPPORTED when a continuous joint has one of the last nj velocity coordinates (q.tail(nj) and the last nj
 * columns would not name the same joints). */
int ikb_problem_add_posture_task(ikb_problem *p, int nj, int priority, const double *weights, const double *mask);
/* CentreOfMassTask (reference centre_of_mass.hpp:14-52, problem.hpp add_centre_of_mass_task, data.cpp:31-34):
 * e = oMr^-1 com(q) - target, J = R_r^T Jcom; 3 rows, target = 3 scalars.  Needs link masses: models from URDF read
 * <inertial><mass>/<origin xyz>; ikb_model_set_inertias supplies them for models built from flat arrays.  Runs on
 * the table-driven kernel unless a loaded plugin matches (ikb_load_specialisation; a plugin folds the model's masses and
 * centres of mass into its code, so it matches only problems whose model still carries those inertias).  Returns the
 * task index (insertion order) or minus an ikb_status. */
int ikb_problem_add_com_task(ikb_problem *p, int ref, int priority, const double *weights /* 3 or NULL */);
/* per joint: mass of the bodies it supports and their centre of mass in the joint frame (Pinocchio inertias[j]) */
int ikb_model_get_inertias(const ikb_model *m, double *mass /* [njoints] */, double *com /* [njoints][3] */);
int ikb_model_set_inertias(ikb_model *m, const double *mass, const double *com);
/* FrameConstraint (reference frame.hpp:333-465; problem.hpp add_frame_constraint): ik::dls projects its step into the null
 * space of the stacked constraint Jacobian, N = I - Jc.completeOrthogonalDecomposition().pseudoInverse() Jc
 * (dls.cpp:26-34,44-52), i.e. keeps `frame` at rest relative to `ref`.  Returns the constraint index or minus an
 * ikb_status.  At most 4 constraints / 12 rows; problems with constraints run on the table-driven kernel unless a loaded
 * plugin generated for the same constraint list matches (ikb_load_specialisation; same count, order, types, frames,
 * reference frames and frame placements). */
int ikb_problem_add_frame_constraint(ikb_problem *p, int frame, int ktype, int ref);
int ikb_problem_c_size(const ikb_problem *p); /* InverseKinematicsProblem::c_size(), problem.hpp:47-53 */
int ikb_problem_num_tasks(const ikb_problem *p);
int ikb_problem_task_dim(const ikb_problem *p, int task);            /* Task::dimension(), task.hpp:38 */
int ikb_problem_e_size(const ikb_problem *p, int priority);          /* problem.hpp:34-40 */
int ikb_problem_rows(const ikb_problem *p);                          /* sum of e_size over levels (dls.hpp:37-41) */
int ikb_problem_target_size(const ikb_problem *p);                   /* scalars of target data per IK problem */
int ikb_problem_task_target_offset(const ikb_problem *p, int task);  /* FRAME: 12 (SE3), ALIGN_AXIS: 3, POSTURE: nj */
/* Upload the problem constants to CUDA device `device` and select the kernel.  After this the handle is immutable. */
int ikb_problem_finalize(ikb_problem *p, int device);
/* Host-only query (no device needed, before or after finalize): name of the compiled topology-specialised kernel
 * that matches this problem's tree and task list exactly, or NULL when the generic table-driven kernel will run. */
const char *ikb_problem_specialisation(const ikb_problem *p);
/* Name of the kernel variant ikb_dls_solve_batch will launch for `dtype` ("coop<...>", "cassie_feet_pelvis", ...) */
const char *ikb_problem_kernel_name(const ikb_problem *p, int dtype);
/* Load a topology-specialised kernel that was generated and compiled AFTER the library was built: a shared object made by
 * `python -m ik_b200.specialise` (tools/gen_kernel.py -> nvcc) for one (URDF, task list) pair.  Problems finalized
 * afterwards that match it exactly take its straight-line kernels instead of the table-driven one -- any robot at the
 * speed of the built-in specialisations.  Also: IKB_SPEC_PLUGINS=a.so:b.so in the environment. */
int ikb_load_specialisation(const char *path);
/* Human-readable note on the kernel selection, "" when there is nothing to say.  A problem that has the topology and
 * task list of a compiled specialisation but whose placements differ from the ones it was generated from (a re-rounded
 * URDF literal, a moved frame) falls back to the table-driven kernel: the note names the specialisation, the first
 * differing joint / frame and the size of the difference, and ikb_problem_finalize prints it once to stderr
 * (IKB_QUIET=1 silences it).  Host-only; valid after ikb_problem_finalize. */
const char *ikb_problem_status_string(const ikb_problem *p);

/* ---- batched solve ------------------------------------------------------------------------------- */
/* Strided views: element k of problem b lives at base[k*elem_stride + b*batch_stride] (strides in elements).
 * SoA batch-major [k][B] is (elem_stride=B, batch_stride=1) -- the coalesced layout the kernels are tuned for;
 * AoS [B][k] is (1, k_count).  batch_stride = 0 broadcasts one vector to the whole batch. */
typedef enum {
    IKB_TARGETS_SE3 = 0,     /* per FrameTask 12 scalars: rotation row-major (9) + translation (3) -- se3_t target, frame.hpp:189 */
    IKB_TARGETS_COMPACT = 1  /* wire format of the HOST entry points, see ikb_problem_compact_target_size */
} ikb_targets_format;

typedef struct {
    const void *q0;      int64_t q0_elem_stride, q0_batch_stride;           /* nq scalars per problem */
    const void *targets; int64_t targets_elem_stride, targets_batch_stride; /* ikb_problem_target_size scalars */
    void *q;             int64_t q_elem_stride, q_batch_stride;             /* result configuration (dls.cpp:63,77) */
    uint8_t *success;  /* [B] problem_data::success (data.hpp:18); may be NULL */
    int32_t *iters;    /* [B] steps taken (dls.cpp:14 loop index at exit); may be NULL */
    void *resid;       /* [B] ||e[0]||^2 at the last evaluation (visitor.hpp:19); may be NULL */
    int32_t targets_format; /* ikb_targets_format; 0 = IKB_TARGETS_SE3.  Zero-initialise the struct (ikb_batch_io io = {0}). */
    int32_t reserved_;
} ikb_batch_io;

/* HOST views (the *_host entry points, ikb_queue_submit_host, ikb_multi_*): q0 / targets / q must be one of
 *   SoA rows      batch_stride 1, elem_stride >= B   (a [k][B] array or a column slice of a wider one),
 *   AoS records   elem_stride 1, batch_stride >= the element count (a [B][k] array or a row slice of a wider one),
 *   a broadcast   batch_stride 0 (inputs only; elem_stride >= 1).
 * Only the payload crosses PCIe (2-D copies skip the gaps of a sliced view); other stridings return
 * IKB_ERR_INVALID_ARG.  DEVICE views (ikb_dls_solve_batch, ikb_queue_submit) may use any strides.
 *
 * Compact targets (IKB_TARGETS_COMPACT): what the reference's callers actually set (ik_ros/src/cassie.cpp:95-99: a
 * translation for a Position task, identity pose for the pelvis) instead of 12 scalars per FrameTask.  Per task, in
 * insertion order: FrameTask Full = unit quaternion x,y,z,w + translation (7 scalars); Position = translation (3;
 * rotation = identity, FrameTask's default target); Orientation = quaternion (4; zero translation); AlignAxisTask,
 * PostureTask and CentreOfMassTask targets are unchanged (3 / nj / 3).  The device expands them to SE3 before the
 * solve (R = quaternion.toRotationMatrix()).  Cassie feet+pelvis: 13 scalars per problem instead of 36. */
int ikb_problem_compact_target_size(const ikb_problem *p);
int ikb_problem_task_compact_target_offset(const ikb_problem *p, int task);

/* Batched ik::dls (reference dls.cpp:5-78 looped over B independent problems).  All pointers in `io` are DEVICE
 * pointers of scalar type `dtype`; the call enqueues on `cuda_stream` (a cudaStream_t, NULL = default stream)
 * and returns without synchronising. */
int ikb_dls_solve_batch(const ikb_problem *p, int dtype, const ikb_dls_params *params, int64_t B,
                        const ikb_batch_io *io, void *cuda_stream);
/* Same with HOST pointers: copies inputs to the device, solves, copies results back and synchronises.  This is
 * the call a user of the reference's API makes; staging buffers are owned by the problem handle.
 * Not re-entrant on one handle (like ik::dls on one dls_data, SURVEY 8b "Threading"). */
int ikb_dls_solve_batch_host(ikb_problem *p, int dtype, const ikb_dls_params *params, int64_t B,
                             const ikb_batch_io *io);
/* vector_t ik::dls(problem, q0, data, visitor, params) for ONE problem in FP64 (reference dls.hpp:111-114):
 * a batch of 1 through the host path. */
int ikb_dls_solve(ikb_problem *p, const ikb_dls_params *params, const double *q0, const double *targets,
                  double *q_out, int *success, int *iters, double *resid);
/* The same, also returning what the reference leaves in its public dls_data / problem_data after the call (data.hpp:15-28,
 * dls.hpp:34-65): dq [nv] = the last step direction computed (dls.cpp:52 -- on success the one at the returned iterate,
 * never applied), e [ikb_problem_rows] = the stacked weighted task errors and J [rows][nv] row-major = the stacked weighted
 * task Jacobian of the last evaluation (dls.cpp:18-24).  Any of the three may be NULL.  Runs on the table-driven
 * team-per-problem kernel (one team, the state is read out of its shared memory), also for problems that have a
 * compiled specialisation; ikb_pik_solve_ex is the ik::pik twin (pik_data, pik.hpp:29-57). */
int ikb_dls_solve_ex(ikb_problem *p, const ikb_dls_params *params, const double *q0, const double *targets,
                     double *q_out, int *success, int *iters, double *resid, double *dq, double *e, double *J);

/* ---- ik::pik: priority-based IK (reference ik/ik/pik.cpp:31-96, pik.hpp:13-57; SURVEY 8f rank 2) ----------------
 * Per iteration: dq = 0, P = I; for every priority level i: de = e_i - J_i dq, Jb = J_i P,
 * dq -= damp_pseudoinverse(Jb, lambda_i) de, P -= Jb.completeOrthogonalDecomposition().pseudoInverse() Jb; then the
 * stop test, integrate and clamp of ik::dls.  (pik_data::da, the null-space bias, is zero in the reference and not
 * exposed.)  Runs on the table-driven kernel for any tree / task mix. */
typedef struct {
    int32_t max_iterations; /* 100 (pik.hpp:14) */
    double step_length;     /* 1.0 (pik.hpp:16) */
    double tolerance;       /* 1e-4 (visitor.hpp:19) */
    /* pik_data::lambda, damping of every priority level: 1.0 (pik.hpp:31).  ik::pik holds at most 7 priority levels:
     * the pik entry points return IKB_ERR_UNSUPPORTED when a task has priority 7 or more (max_priority_level itself
     * may be larger; empty levels above the highest used one cost nothing).  ik::dls takes any priority. */
    double lambda[7];
} ikb_pik_params;
void ikb_pik_params_default(ikb_pik_params *p);
/* as ikb_dls_solve_batch / ikb_dls_solve_batch_host */
int ikb_pik_solve_batch(const ikb_problem *p, int dtype, const ikb_pik_params *params, int64_t B,
                        const ikb_batch_io *io, void *cuda_stream);
int ikb_pik_solve_batch_host(ikb_problem *p, int dtype, const ikb_pik_params *params, int64_t B,
                             const ikb_batch_io *io);
/* vector_t ik::pik(problem, q0, data, visitor, params) for ONE problem in FP64 (pik.hpp:59-66) with the pik_data outputs
 * dq, e, J as ikb_dls_solve_ex (any may be NULL) */
int ikb_pik_solve_ex(ikb_problem *p, const ikb_pik_params *params, const double *q0, const double *targets,
                     double *q_out, int *success, int *iters, double *resid, double *dq, double *e, double *J);

/* ---- pipelined queue --------------------------------------------------------------------------------
 * The reference's only caller runs ik::dls once per control tick, one call after the other
 * (ik_ros/src/cassie.cpp:112-113 inside CassieIK::loop, :146-171).  A stream of BATCHES has the same shape, and one
 * batch alone cannot keep the GPU busy: the few problems that never converge run all max_iterations steps
 * (dls.cpp:14), a serial chain of ~0.7 ms during which most SMs idle.  A queue keeps up to `depth` batches in flight
 * on three internal streams (copy-in, compute, copy-out) and launches `merge` consecutive batches as ONE kernel pair,
 * so the straggler chain is paid once per group and -- with host buffers -- the PCIe copies of one group run beside
 * the kernels of its neighbours.  Batches of a group must share dtype and solver parameters (a change starts a new
 * group).  Results are those of ikb_dls_solve_batch: bit for bit in FP64 whenever both take the same kernels (always
 * for batches larger than the latency configuration holds), to rounding otherwise -- a merged group of small batches
 * may run the thread-per-problem kernels where a lone small batch runs the team-per-problem one, and in FP32 the step
 * at which a straggler changes kernels depends on scheduling.  One thread drives a queue.
 * Groups of device buffers -- and of host buffers when depth >= 3 * merge -- are launched without their own straggler
 * launch: the problems a group's launch suspends (their iterate and step count stay in the batch's own output buffers, for
 * host batches in the slot's staging) continue at the head of the NEXT group's launch, and
 * ikb_queue_wait / _wait_on_stream / _flush / _drain / the reuse of a slot finish them on demand -- a ticket is complete
 * exactly when its wait returns, as before, but two batches in flight must not share output buffers. */
typedef struct ikb_queue ikb_queue;
int ikb_queue_create(ikb_problem *p, int depth /* 1..32 batches in flight */, int merge /* 1..min(depth, 8) */,
                     ikb_queue **out);
void ikb_queue_free(ikb_queue *q);
/* DEVICE buffers (as ikb_dls_solve_batch).  The inputs must be complete in `in_stream` order at the time of the
 * call; the buffers of a batch must stay untouched until its ticket has been waited for.  Returns the batch's
 * ticket (>= 0) or minus an ikb_status.  Blocks only while the slot's previous batch is still in flight. */
int64_t ikb_queue_submit(ikb_queue *q, int dtype, const ikb_dls_params *params, int64_t B, const ikb_batch_io *io,
                         void *in_stream);
/* HOST buffers (as ikb_dls_solve_batch_host; pinned memory -- ikb_host_alloc -- for the copies to overlap). */
int64_t ikb_queue_submit_host(ikb_queue *q, int dtype, const ikb_dls_params *params, int64_t B,
                              const ikb_batch_io *io);
/* Launch the batches submitted so far even if their group is not full. */
int ikb_queue_flush(ikb_queue *q);
/* Block the host until the outputs of `ticket` are complete / make `cuda_stream` wait for them / wait for all.
 * Waiting for a batch whose group is still open launches the group first. */
int ikb_queue_wait(ikb_queue *q, int64_t ticket);
int ikb_queue_wait_on_stream(ikb_queue *q, int64_t ticket, void *cuda_stream);
int ikb_queue_drain(ikb_queue *q);

/* ---- several GPUs behind one handle ------------------------------------------------------------------------
 * north_star: "the batch shards naturally across the 8 GPUs of one box with no NCCL beyond an optional final result
 * gather".  An ikb_multi owns one finalized copy of the problem and one pipelined queue (depth, merge as
 * ikb_queue_create) per listed device; every submitted HOST batch is cut into contiguous slices [r*B/G, (r+1)*B/G)
 * (SURVEY 8e), slice r is copied to, solved on and copied back from device r on that device's own streams -- all
 * devices run concurrently under one host thread -- and the results land directly in the caller's host arrays, so
 * there is no gather step and no collective.  The same device may be listed more than once (its slices then share
 * it).  ikb_multi_gather_device is the optional device-side gather of DEVICE-resident slices onto one GPU
 * (cudaMemcpyPeerAsync over NVLink). */
typedef struct ikb_multi ikb_multi;
int ikb_multi_create(const ikb_problem *p /* not yet finalized, or finalized: it is copied */, const int *devices, int ndevices,
                     int depth, int merge, ikb_multi **out);
void ikb_multi_free(ikb_multi *m);
int ikb_multi_device_count(const ikb_multi *m);
ikb_problem *ikb_multi_problem(ikb_multi *m, int index); /* the finalized per-device copy (for the device-pointer API) */
/* as ikb_queue_submit_host / ikb_queue_wait / ikb_queue_drain; one ticket covers all slices of the batch */
int64_t ikb_multi_submit_host(ikb_multi *m, int dtype, const ikb_dls_params *params, int64_t B, const ikb_batch_io *io);
int ikb_multi_wait(ikb_multi *m, int64_t ticket);
int ikb_multi_drain(ikb_multi *m);
/* blocking: submit + wait (the multi-GPU twin of ikb_dls_solve_batch_host) */
int ikb_multi_dls_solve_batch_host(ikb_multi *m, int dtype, const ikb_dls_params *params, int64_t B, const ikb_batch_io *io);
/* Optional result gather for DEVICE-resident sharded solves (SURVEY 8e): slice r (rows [r*B/G, (r+1)*B/G) of a dense
 * [count][B] SoA array of `elem_bytes`-sized scalars living on device r) is copied into the same rows of `dst` on
 * device `dst_device` with cudaMemcpyPeerAsync on that slice's stream; returns after all copies have completed. */
int ikb_multi_gather_device(ikb_multi *m, const void *const *src /* [ndevices] device pointers, each [count][B_r] */,
                            int count, int64_t B, int elem_bytes, int dst_device, void *dst /* [count][B] */);

/* pinocchio::framesForwardKinematics (reference data.cpp:28-29) for a batch: placements of `nf` frames.
 * q: device, strided as above; out: device SoA [nf*12][B] (frame-major, then the 12 SE3 scalars). */
int ikb_fk_batch(const ikb_problem *p, int dtype, int64_t B, const void *q, int64_t q_elem_stride,
                 int64_t q_batch_stride, int nf, const int32_t *frames, void *out, void *cuda_stream);

/* ---- utilities ------------------------------------------------------------------------------------ */
const char *ikb_last_error(void);
int ikb_version(void);
int ikb_device_count(void);
void *ikb_host_alloc(size_t bytes); /* pinned host memory for the *_host entry points */
void ikb_host_free(void *ptr);
/* FMA-pipe throughput of `device` in TFLOP/s for IKB_F64 / IKB_F32 (mul+add = 2 FLOP): the measured denominator
 * of the compute roofline the IK kernels are judged against (SURVEY.md 8d). */
int ikb_measure_fma_peak(int dtype, int device, double *tflops);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
int64_t ikb_kernel_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* IKB200_H */
