// C ABI of libikb200.so (see include/ikb200.h for the contract and the reference interfaces replaced).
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <climits>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <limits>
#include <memory>
#include <mutex>
#include <type_traits>
#include <stdexcept>
#include <string>
#include <vector>

#include "capi_internal.hpp"
#include "dls_generic.cuh"
#include "problem_fill.hpp"

using namespace ikb;
using namespace ikb::capi;

// ---- definitions of the shared internals (capi_internal.hpp) ----
namespace ikb {
namespace capi {
std::string &last_error() {
    thread_local std::string err;
    return err;
}
std::atomic<long long> g_launches{0};
int fail(int code, const std::string &msg) {
    last_error() = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char *what) {
    return fail(e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? IKB_ERR_NO_DEVICE : IKB_ERR_CUDA,
                std::string(what) + ": " + cudaGetErrorString(e));
}
}  // namespace capi
}  // namespace ikb

namespace {

struct SizeClass {
    int nj, nv, m;
};
const SizeClass kClasses[] = {{10, 8, 6}, {20, 24, 12}, {32, 36, 30}};

template <typename T> DevProblem<T> *dev_blob(const ikb_problem *p);
template <> DevProblem<double> *dev_blob<double>(const ikb_problem *p) { return p->d64; }
template <> DevProblem<float> *dev_blob<float>(const ikb_problem *p) { return p->d32; }

struct FrameList {
    int n;
    int id[16];
};

template <typename T, int NJ>
__global__ void __launch_bounds__(128) fk_model_frames_kernel(const DevProblem<T> *__restrict__ gP, const T *__restrict__ q,
                                                              long long q_es, long long q_bs, long long B, FrameList fl,
                                                              const int *__restrict__ frame_parent,
                                                              const T *__restrict__ frame_placement, T *__restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DevProblem<T> &P = *reinterpret_cast<DevProblem<T> *>(smem_raw);
    unsigned long long *bar = reinterpret_cast<unsigned long long *>(smem_raw + sizeof(DevProblem<T>));
    stage_blob_tma(&P, gP, (unsigned)sizeof(DevProblem<T>), bar);
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    T ql[NJ + 8];
    T oR[NJ][9], op[NJ][3];
    for (int k = 0; k < P.nq; ++k) ql[k] = q[k * q_es + b * q_bs];
    fk_all<T, NJ>(P, ql, oR, op);
    for (int f = 0; f < fl.n; ++f) {
        const int fid = fl.id[f], pj = frame_parent[fid];
        T R[9], p[3];
        se3_mul(oR[pj], op[pj], frame_placement + 12 * fid, frame_placement + 12 * fid + 9, R, p);
#pragma unroll
        for (int i = 0; i < 9; ++i) out[((long long)f * 12 + i) * B + b] = R[i];
#pragma unroll
        for (int i = 0; i < 3; ++i) out[((long long)f * 12 + 9 + i) * B + b] = p[i];
    }
}

template <typename T>
int launch_fk(const ikb_problem *p, int64_t B, const void *q, int64_t es, int64_t bs, const FrameList &fl, void *out,
              cudaStream_t s) {
    const int threads = 128;
    const size_t smem = sizeof(DevProblem<T>) + 16;
    const unsigned blocks = (unsigned)((B + threads - 1) / threads);
    const T *pl = std::is_same<T, double>::value ? (const T *)p->d_frame_pl64 : (const T *)p->d_frame_pl32;
    if (p->size_class <= 1)
        fk_model_frames_kernel<T, 20><<<blocks, threads, smem, s>>>(dev_blob<T>(p), (const T *)q, es, bs, B, fl,
                                                                     p->d_frame_parent, pl, (T *)out);
    else
        fk_model_frames_kernel<T, 32><<<blocks, threads, smem, s>>>(dev_blob<T>(p), (const T *)q, es, bs, B, fl,
                                                                     p->d_frame_parent, pl, (T *)out);
    IKB_CUDA(cudaGetLastError());
    g_launches.fetch_add(1);
    return IKB_OK;
}

// The specialised bodies lay targets out in stacked order, the ABI in insertion order: only problems whose tasks
// were added in non-decreasing priority (stacked order == insertion order) can take the fast path.  A problem with
// FrameConstraints matches only a specialisation generated for the same constraint list (spec_matches).
const SpecializedKernel *select_specialized(const HostProblem &hp) {
    for (size_t i = 1; i < hp.tasks.size(); ++i)
        if (hp.tasks[i].priority < hp.tasks[i - 1].priority) return nullptr;
    return find_specialized(hp);
}

// Compact wire format of the targets (include/ikb200.h), per task in insertion order.
ExpandTable build_expand_table(const HostProblem &hp) {
    ExpandTable t;
    t.ntasks = (int)hp.tasks.size();
    int coff = 0;
    for (int i = 0; i < t.ntasks && i < kMaxTasks; ++i) {
        const HostTask &ht = hp.tasks[i];
        t.toff[i] = hp.target_offset(i);
        t.coff[i] = coff;
        if (ht.kind == IKB_TASK_FRAME) {
            t.mode[i] = ht.type == IKB_FULL ? 1 : (ht.type == IKB_POSITION ? 2 : 3);
            t.n[i] = ht.type == IKB_FULL ? 7 : (ht.type == IKB_POSITION ? 3 : 4);
        } else {
            t.mode[i] = 0;
            t.n[i] = ht.target_size;
        }
        coff += t.n[i];
    }
    t.csz = coff;
    t.tsz = hp.target_size();
    return t;
}

int check_weights(const double *w, int dim, std::vector<double> &out) {
    out.assign(dim, 1.0);
    if (w) std::copy(w, w + dim, out.begin());
    return IKB_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
// exported functions
// ---------------------------------------------------------------------------------------------------
extern "C" {

const char *ikb_last_error(void) { return last_error().c_str(); }
int ikb_version(void) { return IKB_VERSION; }
int64_t ikb_kernel_launch_count(void) { return g_launches.load(); }

int ikb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

void *ikb_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) {
        last_error() = "cudaMallocHost failed";
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void ikb_host_free(void *ptr) {
    if (ptr) cudaFreeHost(ptr);
}

void ikb_dls_params_default(ikb_dls_params *p) {
    if (!p) return;
    p->max_iterations = 100;  // common.hpp:61
    p->random_restart = 0;    // dls.hpp:27
    p->max_time = 1.0;        // common.hpp:63
    p->step_length = 1.0;     // common.hpp:65
    p->damping = 1e-2;        // dls.hpp:25
    p->tolerance = 1e-4;      // visitor.hpp:19
}

int ikb_model_from_urdf(const char *xml, size_t len, int free_flyer, ikb_model **out) {
    if (!xml || !out) return fail(IKB_ERR_INVALID_ARG, "ikb_model_from_urdf: null argument");
    try {
        auto *h = new ikb_model();
        h->m = model_from_urdf(std::string(xml, len), free_flyer != 0);
        *out = h;
        return IKB_OK;
    } catch (const std::exception &e) {
        return fail(IKB_ERR_PARSE, e.what());
    }
}

int ikb_model_from_desc(const ikb_model_desc *d, ikb_model **out) {
    if (!d || !out || d->njoints < 1 || !d->parent || !d->jtype || !d->placement)
        return fail(IKB_ERR_INVALID_ARG, "ikb_model_from_desc: null / empty description");
    if (d->jtype[0] != IKB_J_UNIVERSE) return fail(IKB_ERR_INVALID_ARG, "joint 0 must be the universe");
    auto *h = new ikb_model();
    HostModel &m = h->m;
    int iq = 0;
    for (int j = 0; j < d->njoints; ++j) {
        const int t = d->jtype[j];
        if (t < IKB_J_UNIVERSE || t > IKB_J_RUB_UNALIGNED || (j > 0 && (d->parent[j] < 0 || d->parent[j] >= j))) {
            delete h;
            return fail(IKB_ERR_INVALID_ARG, "ikb_model_from_desc: bad joint type or parent index (parents must precede children)");
        }
        SE3d pl;
        std::copy(d->placement + 12 * j, d->placement + 12 * j + 12, pl.begin());
        std::array<double, 3> ax{0, 0, 0};
        if (d->axis) ax = {d->axis[3 * j], d->axis[3 * j + 1], d->axis[3 * j + 2]};
        const int n = joint_nq(t);
        std::vector<double> lo(n), hi(n);
        for (int k = 0; k < n; ++k) {
            lo[k] = d->lower ? d->lower[iq + k] : -1e300;
            hi[k] = d->upper ? d->upper[iq + k] : 1e300;
        }
        iq += n;
        m.add_joint(d->joint_names && d->joint_names[j] ? d->joint_names[j] : ("joint" + std::to_string(j)), t,
                    j == 0 ? 0 : d->parent[j], pl, ax, lo, hi);
    }
    for (int f = 0; f < d->nframes; ++f) {
        if (d->frame_parent[f] < 0 || d->frame_parent[f] >= d->njoints) {
            delete h;
            return fail(IKB_ERR_INVALID_ARG, "ikb_model_from_desc: frame parent out of range");
        }
        SE3d pl;
        std::copy(d->frame_placement + 12 * f, d->frame_placement + 12 * f + 12, pl.begin());
        m.add_frame(d->frame_names && d->frame_names[f] ? d->frame_names[f] : ("frame" + std::to_string(f)),
                    d->frame_parent[f], pl, FRAME_OP);
    }
    if (m.nframes() == 0) m.add_frame("universe", 0, se3_identity(), FRAME_OP);
    *out = h;
    return IKB_OK;
}

void ikb_model_free(ikb_model *m) { delete m; }
int ikb_model_njoints(const ikb_model *m) { return m ? m->m.njoints() : -IKB_ERR_INVALID_ARG; }
int ikb_model_nq(const ikb_model *m) { return m ? m->m.nq : -IKB_ERR_INVALID_ARG; }
int ikb_model_nv(const ikb_model *m) { return m ? m->m.nv : -IKB_ERR_INVALID_ARG; }
int ikb_model_nframes(const ikb_model *m) { return m ? m->m.nframes() : -IKB_ERR_INVALID_ARG; }
int ikb_model_frame_id(const ikb_model *m, const char *name) {
    if (!m || !name) return -IKB_ERR_INVALID_ARG;
    return m->m.frame_id(name);
}
const char *ikb_model_joint_name(const ikb_model *m, int j) {
    return (m && j >= 0 && j < m->m.njoints()) ? m->m.joint_names[j].c_str() : nullptr;
}
const char *ikb_model_frame_name(const ikb_model *m, int f) {
    return (m && f >= 0 && f < m->m.nframes()) ? m->m.frame_names[f].c_str() : nullptr;
}
int ikb_model_get_topology(const ikb_model *m, int32_t *parent, int32_t *jtype, int32_t *idx_q, int32_t *idx_v) {
    if (!m) return fail(IKB_ERR_INVALID_ARG, "null model");
    const int n = m->m.njoints();
    if (parent) std::copy(m->m.parent.begin(), m->m.parent.end(), parent);
    if (jtype) std::copy(m->m.jtype.begin(), m->m.jtype.end(), jtype);
    if (idx_q) std::copy(m->m.idx_q.begin(), m->m.idx_q.end(), idx_q);
    if (idx_v) std::copy(m->m.idx_v.begin(), m->m.idx_v.end(), idx_v);
    (void)n;
    return IKB_OK;
}
int ikb_model_get_placements(const ikb_model *m, double *placement, double *axis) {
    if (!m) return fail(IKB_ERR_INVALID_ARG, "null model");
    for (int j = 0; j < m->m.njoints(); ++j) {
        if (placement) std::copy(m->m.placement[j].begin(), m->m.placement[j].end(), placement + 12 * j);
        if (axis) std::copy(m->m.axis[j].begin(), m->m.axis[j].end(), axis + 3 * j);
    }
    return IKB_OK;
}
int ikb_model_get_limits(const ikb_model *m, double *lower, double *upper) {
    if (!m) return fail(IKB_ERR_INVALID_ARG, "null model");
    if (lower) std::copy(m->m.lower.begin(), m->m.lower.end(), lower);
    if (upper) std::copy(m->m.upper.begin(), m->m.upper.end(), upper);
    return IKB_OK;
}
int ikb_model_set_limits(ikb_model *m, const double *lower, const double *upper) {
    if (!m) return fail(IKB_ERR_INVALID_ARG, "null model");
    if (lower) std::copy(lower, lower + m->m.nq, m->m.lower.begin());
    if (upper) std::copy(upper, upper + m->m.nq, m->m.upper.begin());
    return IKB_OK;
}
int ikb_model_get_frames(const ikb_model *m, int32_t *parent_joint, int32_t *type, double *placement) {
    if (!m) return fail(IKB_ERR_INVALID_ARG, "null model");
    for (int f = 0; f < m->m.nframes(); ++f) {
        if (parent_joint) parent_joint[f] = m->m.frame_parent[f];
        if (type) type[f] = m->m.frame_type[f];
        if (placement) std::copy(m->m.frame_placement[f].begin(), m->m.frame_placement[f].end(), placement + 12 * f);
    }
    return IKB_OK;
}
int ikb_model_neutral(const ikb_model *m, double *q) {
    if (!m || !q) return fail(IKB_ERR_INVALID_ARG, "null argument");
    std::fill(q, q + m->m.nq, 0.0);
    for (int j = 0; j < m->m.njoints(); ++j)
        if (m->m.jtype[j] == IKB_J_FREEFLYER) q[m->m.idx_q[j] + 6] = 1.0;
        else if (is_continuous(m->m.jtype[j])) q[m->m.idx_q[j]] = 1.0;   // (cos, sin) = (1, 0)
    return IKB_OK;
}

int ikb_problem_create(const ikb_model *m, int max_priority_level, ikb_problem **out) {
    if (!m || !out || max_priority_level < 0) return fail(IKB_ERR_INVALID_ARG, "ikb_problem_create: bad argument");
    auto *p = new ikb_problem();
    p->hp.model = m->m;  // copy, like InverseKinematicsProblem (problem.hpp:183)
    p->hp.max_priority_level = max_priority_level;
    *out = p;
    return IKB_OK;
}

void ikb_problem_free(ikb_problem *p) {
    if (!p) return;
    if (p->device >= 0) {   // device state may be partially built when ikb_problem_finalize failed half-way: free whatever exists
        DeviceGuard g(p->device);
        cudaFree(p->d64); cudaFree(p->d32); cudaFree(p->d_frame_parent); cudaFree(p->d_frame_pl64);
        cudaFree(p->d_frame_pl32); cudaFree(p->d_tickets);
        cudaFree(p->st64.q0); cudaFree(p->st64.targets); cudaFree(p->st64.q); cudaFree(p->st64.resid); cudaFree(p->st64.compact);
        cudaFree(p->st32.q0); cudaFree(p->st32.targets); cudaFree(p->st32.q); cudaFree(p->st32.resid); cudaFree(p->st32.compact);
        cudaFree(p->st_success); cudaFree(p->st_iters); cudaFree(p->st_aux);
        for (auto &sc : p->scratch) {
            cudaFree(sc.list); cudaFree(sc.iters);
            if (sc.ev) cudaEventDestroy(sc.ev);
        }
        for (void *r : p->retired) cudaFree(r);
        for (auto e : p->ticket_ev) if (e) cudaEventDestroy(e);
        if (p->stream) cudaStreamDestroy(p->stream);
        if (p->stream_in) cudaStreamDestroy(p->stream_in);
        if (p->stream_aux) cudaStreamDestroy(p->stream_aux);
        for (auto e : p->ev_in) if (e) cudaEventDestroy(e);
        if (p->ev_aux) cudaEventDestroy(p->ev_aux);
        if (p->ev_main) cudaEventDestroy(p->ev_main);
    }
    delete p;
}

static int add_task_common(ikb_problem *p, HostTask &t, int priority, const double *weights) {
    if (p->finalized) return -fail(IKB_ERR_INVALID_ARG, "problem is finalized (immutable)");
    if (priority < 0 || priority > p->hp.max_priority_level)
        return -fail(IKB_ERR_INVALID_ARG, "priority exceeds max_priority_level (problem.hpp:160-164)");
    t.priority = priority;
    check_weights(weights, t.dim, t.weight);
    p->hp.tasks.push_back(t);
    return (int)p->hp.tasks.size() - 1;
}

int ikb_problem_add_frame_task(ikb_problem *p, int frame, int ktype, int ref, int priority, const double *weights) {
    if (!p) return -fail(IKB_ERR_INVALID_ARG, "null problem");
    const int nf = p->hp.model.nframes();
    if (frame < 0 || frame >= nf || ref < 0 || ref >= nf) return -fail(IKB_ERR_UNKNOWN_FRAME, "frame index out of range");
    if (ktype < IKB_POSITION || ktype > IKB_FULL) return -fail(IKB_ERR_INVALID_ARG, "bad kinematic type");
    HostTask t;
    t.kind = IKB_TASK_FRAME;
    t.frame = frame;
    t.ref = ref;
    t.type = ktype;
    t.dim = ktype == IKB_FULL ? 6 : 3;  // frame.hpp:100-107
    t.target_size = 12;
    return add_task_common(p, t, priority, weights);
}

int ikb_problem_add_align_axis_task(ikb_problem *p, int frame, int axis, int ref, int priority, const double *weights) {
    if (!p) return -fail(IKB_ERR_INVALID_ARG, "null problem");
    const int nf = p->hp.model.nframes();
    if (frame < 0 || frame >= nf || ref < 0 || ref >= nf) return -fail(IKB_ERR_UNKNOWN_FRAME, "frame index out of range");
    if (axis < 0 || axis > 2) return -fail(IKB_ERR_INVALID_ARG, "bad axis");
    HostTask t;
    t.kind = IKB_TASK_ALIGN_AXIS;
    t.frame = frame;
    t.ref = ref;
    t.type = axis;
    t.dim = 1;  // frame.hpp:226
    t.target_size = 3;
    return add_task_common(p, t, priority, weights);
}

int ikb_problem_add_posture_task(ikb_problem *p, int nj, int priority, const double *weights, const double *mask) {
    if (!p) return -fail(IKB_ERR_INVALID_ARG, "null problem");
    const HostModel &m = p->hp.model;
    if (nj < 1 || nj > m.nv || nj > m.nq) return -fail(IKB_ERR_INVALID_ARG, "posture size out of range");
    // posture.hpp:50-67 pairs q.tail(nj) with the last nj velocity coordinates: with a continuous joint (two entries of q,
    // one of v) among those, they no longer name the same joints
    for (int j = 1; j < m.njoints(); ++j)
        if (is_continuous(m.jtype[j]) && m.idx_v[j] >= m.nv - nj)
            return -fail(IKB_ERR_UNSUPPORTED, "posture task over the last " + std::to_string(nj) + " coordinates: joint " +
                                                  m.joint_names[j] + " among them is continuous, so q.tail(nj) and the last nj "
                                                  "velocity coordinates would not name the same joints");
    HostTask t;
    t.kind = IKB_TASK_POSTURE;
    t.type = nj;
    t.dim = nj;  // posture.hpp:32
    t.target_size = nj;
    t.mask.assign(nj, 1.0);
    if (mask) std::copy(mask, mask + nj, t.mask.begin());
    return add_task_common(p, t, priority, weights);
}

int ikb_problem_add_com_task(ikb_problem *p, int ref, int priority, const double *weights) {
    if (!p) return -fail(IKB_ERR_INVALID_ARG, "null problem");
    if (ref < 0 || ref >= p->hp.model.nframes()) return -fail(IKB_ERR_UNKNOWN_FRAME, "frame index out of range");
    double tm = 0;
    for (int j = 1; j < p->hp.model.njoints(); ++j) tm += p->hp.model.mass[j];
    if (!(tm > 0)) return -fail(IKB_ERR_INVALID_ARG, "the model carries no mass (no <inertial> in the URDF / ikb_model_set_inertias)");
    HostTask t;
    t.kind = IKB_TASK_COM;
    t.frame = ref;
    t.ref = ref;
    t.type = 0;
    t.dim = 3;
    t.target_size = 3;
    return add_task_common(p, t, priority, weights);
}

int ikb_model_get_inertias(const ikb_model *m, double *mass, double *com) {
    if (!m) return fail(IKB_ERR_INVALID_ARG, "null model");
    for (int j = 0; j < m->m.njoints(); ++j) {
        if (mass) mass[j] = m->m.mass[j];
        if (com)
            for (int k = 0; k < 3; ++k) com[3 * j + k] = m->m.com[j][k];
    }
    return IKB_OK;
}
int ikb_model_set_inertias(ikb_model *m, const double *mass, const double *com) {
    if (!m || !mass || !com) return fail(IKB_ERR_INVALID_ARG, "null argument");
    for (int j = 0; j < m->m.njoints(); ++j) {
        if (!(mass[j] >= 0)) return fail(IKB_ERR_INVALID_ARG, "negative mass");
        m->m.mass[j] = mass[j];
        for (int k = 0; k < 3; ++k) m->m.com[j][k] = com[3 * j + k];
    }
    return IKB_OK;
}

int ikb_problem_add_frame_constraint(ikb_problem *p, int frame, int ktype, int ref) {
    if (!p) return -fail(IKB_ERR_INVALID_ARG, "null problem");
    if (p->finalized) return -fail(IKB_ERR_INVALID_ARG, "problem is finalized (immutable)");
    const int nf = p->hp.model.nframes();
    if (frame < 0 || frame >= nf || ref < 0 || ref >= nf) return -fail(IKB_ERR_UNKNOWN_FRAME, "frame index out of range");
    if (ktype != IKB_POSITION && ktype != IKB_ORIENTATION && ktype != IKB_FULL)
        return -fail(IKB_ERR_INVALID_ARG, "kinematic type must be IKB_POSITION, IKB_ORIENTATION or IKB_FULL");
    HostConstraint c;
    c.frame = frame;
    c.ref = ref;
    c.type = ktype;
    c.dim = ktype == IKB_FULL ? 6 : 3;
    p->hp.constraints.push_back(c);
    return (int)p->hp.constraints.size() - 1;
}
int ikb_problem_c_size(const ikb_problem *p) { return p ? p->hp.c_size() : -IKB_ERR_INVALID_ARG; }

int ikb_problem_num_tasks(const ikb_problem *p) { return p ? (int)p->hp.tasks.size() : -IKB_ERR_INVALID_ARG; }
int ikb_problem_task_dim(const ikb_problem *p, int t) {
    return (p && t >= 0 && t < (int)p->hp.tasks.size()) ? p->hp.tasks[t].dim : -IKB_ERR_INVALID_ARG;
}
int ikb_problem_e_size(const ikb_problem *p, int priority) { return p ? p->hp.e_size(priority) : -IKB_ERR_INVALID_ARG; }
int ikb_problem_rows(const ikb_problem *p) { return p ? p->hp.rows() : -IKB_ERR_INVALID_ARG; }
int ikb_problem_target_size(const ikb_problem *p) { return p ? p->hp.target_size() : -IKB_ERR_INVALID_ARG; }
int ikb_problem_task_target_offset(const ikb_problem *p, int t) {
    return (p && t >= 0 && t < (int)p->hp.tasks.size()) ? p->hp.target_offset(t) : -IKB_ERR_INVALID_ARG;
}

int ikb_problem_finalize(ikb_problem *p, int device) {
    if (!p) return fail(IKB_ERR_INVALID_ARG, "null problem");
    if (p->finalized) return fail(IKB_ERR_INVALID_ARG, "problem already finalized");
    const HostProblem &hp = p->hp;
    const HostModel &m = hp.model;
    if (hp.tasks.empty()) return fail(IKB_ERR_INVALID_ARG, "problem has no tasks");
    const std::vector<int> order = stacked_order(hp);
    const std::vector<int> used = used_frames(hp);
    if ((int)hp.constraints.size() > kMaxConstraints || hp.c_size() > kMaxConstraintRows)
        return fail(IKB_ERR_UNSUPPORTED, "at most 4 frame constraints / 12 constraint rows");
    if (m.njoints() > kMaxJoints || m.nq > kMaxNq || (int)hp.tasks.size() > kMaxTasks || (int)used.size() > kMaxFrames ||
        hp.rows() > kMaxRows)
        return fail(IKB_ERR_UNSUPPORTED, "problem exceeds the compiled capacities of the constant blob");
    int cls = -1;
    for (int c = 0; c < 3; ++c)   // the kernels size q as nv + 4 scalars (continuous joints make nq exceed nv)
        if (m.njoints() <= kClasses[c].nj && m.nv <= kClasses[c].nv && m.nq <= kClasses[c].nv + 4 && hp.rows() <= kClasses[c].m) {
            cls = c;
            break;
        }
    if (cls < 0)
        return fail(IKB_ERR_UNSUPPORTED, "problem larger than the generic kernel's largest size class (32 joints, nv 36, nq 40, 30 rows)");

    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(IKB_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
    }
    if (device < 0 || device >= ndev) return fail(IKB_ERR_INVALID_ARG, "device index out of range");
    DeviceGuard g(device);
    if (!g.ok) return fail(IKB_ERR_CUDA, "cudaSetDevice failed");
    cudaDeviceProp prop;
    IKB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(IKB_ERR_NO_DEVICE, std::string("device ") + prop.name + " is not Blackwell-class (sm_100a code only)");
    p->device = device;   // from here on ikb_problem_free releases whatever device state exists
    p->sm_count = prop.multiProcessorCount;
    if (const char *e = std::getenv("IKB_SM_LIMIT")) {  // measurement knob: persistent grids sized for fewer SMs (read at finalize)
        const int lim = std::atoi(e);
        if (lim >= 1 && lim < p->sm_count) p->sm_count = lim;
    }

    {
        std::unique_ptr<DevProblem<double>> h64(new DevProblem<double>());
        std::unique_ptr<DevProblem<float>> h32(new DevProblem<float>());
        fill_dev_problem(hp, order, used, *h64);
        fill_dev_problem(hp, order, used, *h32);
        p->coop_ok = h64->coop_ok != 0;
        IKB_CUDA(cudaMalloc(&p->d64, sizeof(*h64)));
        IKB_CUDA(cudaMalloc(&p->d32, sizeof(*h32)));
        IKB_CUDA(cudaMemcpy(p->d64, h64.get(), sizeof(*h64), cudaMemcpyHostToDevice));
        IKB_CUDA(cudaMemcpy(p->d32, h32.get(), sizeof(*h32), cudaMemcpyHostToDevice));
    }

    const int nf = m.nframes();
    std::vector<double> pl64((size_t)nf * 12);
    std::vector<float> pl32((size_t)nf * 12);
    for (int f = 0; f < nf; ++f)
        for (int k = 0; k < 12; ++k) {
            pl64[12 * f + k] = m.frame_placement[f][k];
            pl32[12 * f + k] = (float)m.frame_placement[f][k];
        }
    IKB_CUDA(cudaMalloc(&p->d_frame_parent, nf * sizeof(int)));
    IKB_CUDA(cudaMalloc(&p->d_frame_pl64, pl64.size() * sizeof(double)));
    IKB_CUDA(cudaMalloc(&p->d_frame_pl32, pl32.size() * sizeof(float)));
    IKB_CUDA(cudaMemcpy(p->d_frame_parent, m.frame_parent.data(), nf * sizeof(int), cudaMemcpyHostToDevice));
    IKB_CUDA(cudaMemcpy(p->d_frame_pl64, pl64.data(), pl64.size() * sizeof(double), cudaMemcpyHostToDevice));
    IKB_CUDA(cudaMemcpy(p->d_frame_pl32, pl32.data(), pl32.size() * sizeof(float), cudaMemcpyHostToDevice));
    IKB_CUDA(cudaMalloc(&p->d_tickets, kTicketSlots * 16 * sizeof(unsigned long long)));
    IKB_CUDA(cudaMemset(p->d_tickets, 0, kTicketSlots * 16 * sizeof(unsigned long long)));
    for (auto &e : p->ticket_ev) IKB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    IKB_CUDA(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    IKB_CUDA(cudaStreamCreateWithFlags(&p->stream_in, cudaStreamNonBlocking));
    IKB_CUDA(cudaStreamCreateWithFlags(&p->stream_aux, cudaStreamNonBlocking));
    for (auto &e : p->ev_in) IKB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    IKB_CUDA(cudaEventCreateWithFlags(&p->ev_aux, cudaEventDisableTiming));
    IKB_CUDA(cudaEventCreateWithFlags(&p->ev_main, cudaEventDisableTiming));

    p->size_class = cls;
    p->expand = build_expand_table(hp);
    p->weight_stacked.clear();
    p->mask_stacked.clear();
    for (int t : order) {
        for (double w : hp.tasks[t].weight) p->weight_stacked.push_back(w);
        for (int i = 0; i < hp.tasks[t].dim; ++i)
            p->mask_stacked.push_back(hp.tasks[t].kind == IKB_TASK_POSTURE ? hp.tasks[t].mask[i] : 1.0);
    }
    p->spec = select_specialized(hp);
    p->status.clear();
    if (!p->spec) {
        const char *forced = std::getenv("IKB_FORCE_GENERIC");
        std::string why;
        if (!(forced && forced[0] == '1') && find_near_miss(hp, &why)) {
            p->status = why;
            const char *quiet = std::getenv("IKB_QUIET");
            static std::atomic<bool> warned{false};
            if (!(quiet && quiet[0] == '1') && !warned.exchange(true)) std::fprintf(stderr, "[ikb200] %s\n", why.c_str());
        }
    }
    char buf[96];
    const char *legacy = std::getenv("IKB_GENERIC_LEGACY");
    const int team[3] = {8, 16, 32};
    if (p->coop_ok && !(legacy && legacy[0] == '1')) {
        p->size_class = cls;   // (coop_class reads it)
        const int cc = coop_class(p);   // a class-2 problem on a Cassie-sized tree runs with class 1's tree capacities
        std::snprintf(buf, sizeof buf, "coop<NJ=%d,NV=%d,M=%d,TEAM=%d>", kClasses[cc == 3 ? 1 : cls].nj, kClasses[cc == 3 ? 1 : cls].nv, kClasses[cls].m, team[cls]);
    }
    else
        std::snprintf(buf, sizeof buf, "generic<NJ=%d,NV=%d,M=%d>", kClasses[cls].nj, kClasses[cls].nv, kClasses[cls].m);
    p->kernel_name[0] = p->spec ? p->spec->name : buf;
    p->kernel_name[1] = p->kernel_name[0];
    p->finalized = true;
    return IKB_OK;
}

const char *ikb_problem_specialisation(const ikb_problem *p) {
    if (!p || p->hp.tasks.empty()) return nullptr;
    const SpecializedKernel *k = select_specialized(p->hp);
    return k ? k->name : nullptr;
}

int ikb_load_specialisation(const char *path) {
    if (!path) return fail(IKB_ERR_INVALID_ARG, "null path");
    std::string err;
    if (load_specialisation_plugin(path, &err)) return fail(IKB_ERR_INVALID_ARG, err);
    return IKB_OK;
}

const char *ikb_problem_status_string(const ikb_problem *p) { return p ? p->status.c_str() : ""; }

int ikb_problem_compact_target_size(const ikb_problem *p) { return p ? build_expand_table(p->hp).csz : -IKB_ERR_INVALID_ARG; }
int ikb_problem_task_compact_target_offset(const ikb_problem *p, int t) {
    if (!p || t < 0 || t >= (int)p->hp.tasks.size()) return -IKB_ERR_INVALID_ARG;
    return build_expand_table(p->hp).coff[t];
}

const char *ikb_problem_kernel_name(const ikb_problem *p, int dtype) {
    if (!p || !p->finalized || dtype < 0 || dtype > 1) return nullptr;
    return p->kernel_name[dtype].c_str();
}

int ikb_fk_batch(const ikb_problem *p, int dtype, int64_t B, const void *q, int64_t es, int64_t bs, int nf,
                 const int32_t *frames, void *out, void *cuda_stream) {
    if (!p || !q || !out || !frames) return fail(IKB_ERR_INVALID_ARG, "null argument");
    if (!p->finalized) return fail(IKB_ERR_NOT_FINALIZED, "call ikb_problem_finalize first");
    if (nf < 1 || nf > 16) return fail(IKB_ERR_INVALID_ARG, "between 1 and 16 frames per call");
    FrameList fl;
    fl.n = nf;
    for (int i = 0; i < nf; ++i) {
        if (frames[i] < 0 || frames[i] >= p->hp.model.nframes()) return fail(IKB_ERR_UNKNOWN_FRAME, "frame index out of range");
        fl.id[i] = frames[i];
    }
    if (B <= 0) return IKB_OK;
    DeviceGuard g(p->device);
    cudaStream_t s = (cudaStream_t)cuda_stream;
    return dtype == IKB_F64 ? launch_fk<double>(p, B, q, es, bs, fl, out, s) : launch_fk<float>(p, B, q, es, bs, fl, out, s);
}

}  // extern "C"
