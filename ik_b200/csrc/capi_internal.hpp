// Internals shared by the translation units of the C ABI (ikb_capi.cu: models, problems, FK, utilities; ikb_solve.cu:
// the solve launcher and the host-buffer path; ikb_queue.cu: the pipelined queue).  Not installed; include/ikb200.h is
// the public contract.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <climits>
#include <cstdint>
#include <cstdlib>
#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/ikb200.h"
#include "dev_problem.hpp"
#include "model.hpp"
#include "specialized.hpp"

namespace ikb {
namespace capi {
constexpr int kTicketSlots = 64;
constexpr int kScratchSlots = 8;

// Device scratch of one in-flight two-phase solve: the suspended-problem list and (when the caller passes no `iters`)
// the step counts the tail launch resumes from.  Slots rotate; `ev` marks the end of the slot's last user.
struct SolveScratch {
    unsigned int *list = nullptr;
    int *iters = nullptr;
    size_t cap = 0;
    cudaEvent_t ev = nullptr;
};

// Device staging buffers of one host-buffer batch (same strides as the caller's views).
template <typename T> struct Staging {
    T *q0 = nullptr, *targets = nullptr, *q = nullptr, *resid = nullptr;
    size_t q0_cap = 0, tg_cap = 0, q_cap = 0, b_cap = 0;
    T *compact = nullptr;  // IKB_TARGETS_COMPACT: the wire-format targets as copied in; `targets` receives the SE3 expansion
    size_t compact_cap = 0;
};

// Compact wire format of the targets (include/ikb200.h): per task (insertion order) what to expand and where.
struct ExpandTable {
    int ntasks = 0;
    int mode[kMaxTasks] = {};   // 0: copy `n` scalars; 1: quaternion + translation -> SE3; 2: translation -> (I, p); 3: quaternion -> (R, 0)
    int n[kMaxTasks] = {};
    int coff[kMaxTasks] = {};   // offset in the compact record
    int toff[kMaxTasks] = {};   // offset in the SE3 record
    int csz = 0, tsz = 0;
};
}  // namespace capi
}  // namespace ikb

struct ikb_model {
    ikb::HostModel m;
};

struct ikb_problem {
    ikb::HostProblem hp;
    bool finalized = false;
    int device = -1;
    int size_class = -1;
    bool coop_ok = false;   // the team-per-problem kernel's tables fit (dls_coop.cuh); else the thread-per-problem fallback
    int sm_count = 0;
    ikb::DevProblem<double> *d64 = nullptr;
    ikb::DevProblem<float> *d32 = nullptr;
    int *d_frame_parent = nullptr;  // all model frames (for ikb_fk_batch)
    double *d_frame_pl64 = nullptr;
    float *d_frame_pl32 = nullptr;
    unsigned long long *d_tickets = nullptr;
    std::atomic<unsigned> ticket_next{0};
    cudaEvent_t ticket_ev[ikb::capi::kTicketSlots] = {};  // end of the last launch that used the slot's counters (any stream)
    ikb::capi::SolveScratch scratch[ikb::capi::kScratchSlots];
    std::vector<void *> retired;   // scratch buffers replaced by larger ones: freed with the handle, never while in flight
    std::mutex scratch_mu;
    ikb::capi::ExpandTable expand;
    std::string status;            // ikb_problem_status_string
    const ikb::SpecializedKernel *spec = nullptr;
    std::vector<double> weight_stacked;  // Task::weighting() rows in stacked order (constants of the specialised kernels)
    std::vector<double> mask_stacked;    // posture masks per row, 1 for the rows of other tasks
    std::string kernel_name[2];
    // host-path staging (ikb_dls_solve_batch_host): main stream + the pipelined path's copy-in and second compute stream
    cudaStream_t stream = nullptr, stream_in = nullptr, stream_aux = nullptr;
    cudaEvent_t ev_in[8] = {}, ev_aux = nullptr, ev_main = nullptr;
    ikb::capi::Staging<double> st64;
    ikb::capi::Staging<float> st32;
    unsigned char *st_success = nullptr;
    int *st_iters = nullptr;
    size_t st_flag_cap = 0;
    void *st_aux = nullptr;   // dq / e / J of the *_solve_ex calls (host path only; grown on demand)
    size_t st_aux_cap = 0;
};

namespace ikb {
namespace capi {

// ---- error reporting (ikb_last_error is per thread) ----
std::string &last_error();
extern std::atomic<long long> g_launches;
int fail(int code, const std::string &msg);
int cuda_fail(cudaError_t e, const char *what);
#define IKB_CUDA(call)                                                  \
    do {                                                                \
        cudaError_t e_ = (call);                                        \
        if (e_ != cudaSuccess) return ::ikb::capi::cuda_fail(e_, #call); \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

int check_solve_args(const ikb_problem *p, int dtype, const ikb_dls_params *prm, int64_t B, const ikb_batch_io *io);

// ---- buffers ----
inline size_t view_extent(int64_t n_elem, int64_t es, int64_t bs, int64_t B) {
    return (size_t)((n_elem - 1) * es + (B - 1) * bs + 1);
}

// HOST views (include/ikb200.h): SoA rows, AoS records or a broadcast.  The device staging copy is always DENSE in the
// same orientation -- only the payload crosses PCIe, whatever gaps the caller's view has.
enum ViewKind { VIEW_SOA = 0, VIEW_AOS = 1, VIEW_BCAST = 2, VIEW_BAD = 3 };
struct HostView {
    const void *base = nullptr;
    long long es = 0, bs = 0;
    int n = 0;
    ViewKind kind = VIEW_BAD;
    // strides of the dense device copy
    long long dev_es(long long B) const { return kind == VIEW_SOA ? B : 1; }
    long long dev_bs() const { return kind == VIEW_SOA ? 1 : (kind == VIEW_AOS ? n : 0); }
    size_t dev_count(long long B) const { return kind == VIEW_BCAST ? (size_t)n : (size_t)n * (size_t)B; }
};
inline HostView host_view(const void *base, long long es, long long bs, int n, long long B, bool input) {
    HostView v;
    v.base = base; v.es = es; v.bs = bs; v.n = n;
    if (n <= 0) v.kind = VIEW_AOS;
    else if (bs == 0) v.kind = (input && es >= 1) ? VIEW_BCAST : VIEW_BAD;
    else if (es == 1 && bs >= n) v.kind = VIEW_AOS;
    else if (bs == 1 && es >= B) v.kind = VIEW_SOA;
    else v.kind = VIEW_BAD;
    return v;
}
// Host -> device copy of batch slice [b0, b1) of `v` into its dense staging copy `dst` (`first`: broadcasts travel once).
template <typename T> int copy_view_in(T *dst, const HostView &v, long long B, long long b0, long long b1, bool first, cudaStream_t s) {
    if (v.n <= 0 || b1 <= b0) return IKB_OK;
    const T *src = (const T *)v.base;
    if (v.kind == VIEW_BCAST) {
        if (!first) return IKB_OK;
        if (v.es == 1) IKB_CUDA(cudaMemcpyAsync(dst, src, (size_t)v.n * sizeof(T), cudaMemcpyHostToDevice, s));
        else IKB_CUDA(cudaMemcpy2DAsync(dst, sizeof(T), src, (size_t)v.es * sizeof(T), sizeof(T), (size_t)v.n, cudaMemcpyHostToDevice, s));
    } else if (v.kind == VIEW_SOA) {
        if (v.es == B && b0 == 0 && b1 == B) IKB_CUDA(cudaMemcpyAsync(dst, src, (size_t)v.n * (size_t)B * sizeof(T), cudaMemcpyHostToDevice, s));
        else IKB_CUDA(cudaMemcpy2DAsync(dst + b0, (size_t)B * sizeof(T), src + b0, (size_t)v.es * sizeof(T), (size_t)(b1 - b0) * sizeof(T),
                                        (size_t)v.n, cudaMemcpyHostToDevice, s));
    } else {
        if (v.bs == v.n) IKB_CUDA(cudaMemcpyAsync(dst + b0 * v.n, src + b0 * v.n, (size_t)(b1 - b0) * v.n * sizeof(T), cudaMemcpyHostToDevice, s));
        else IKB_CUDA(cudaMemcpy2DAsync(dst + b0 * v.n, (size_t)v.n * sizeof(T), src + b0 * v.bs, (size_t)v.bs * sizeof(T), (size_t)v.n * sizeof(T),
                                        (size_t)(b1 - b0), cudaMemcpyHostToDevice, s));
    }
    return IKB_OK;
}
// Device -> host copy of the dense staging copy `src` into the caller's view.
template <typename T> int copy_view_out(const HostView &v, const T *src, long long B, cudaStream_t s) {
    if (v.n <= 0 || B <= 0) return IKB_OK;
    T *dst = (T *)v.base;
    if (v.kind == VIEW_SOA) {
        if (v.es == B) IKB_CUDA(cudaMemcpyAsync(dst, src, (size_t)v.n * (size_t)B * sizeof(T), cudaMemcpyDeviceToHost, s));
        else IKB_CUDA(cudaMemcpy2DAsync(dst, (size_t)v.es * sizeof(T), src, (size_t)B * sizeof(T), (size_t)B * sizeof(T), (size_t)v.n, cudaMemcpyDeviceToHost, s));
    } else {
        if (v.bs == v.n) IKB_CUDA(cudaMemcpyAsync(dst, src, (size_t)v.n * (size_t)B * sizeof(T), cudaMemcpyDeviceToHost, s));
        else IKB_CUDA(cudaMemcpy2DAsync(dst, (size_t)v.bs * sizeof(T), src, (size_t)v.n * sizeof(T), (size_t)v.n * sizeof(T), (size_t)B, cudaMemcpyDeviceToHost, s));
    }
    return IKB_OK;
}

// The three views of a host batch, classified; IKB_ERR_INVALID_ARG for stridings the host entry points do not take.
struct HostViews {
    HostView q0, tg, q;
    bool compact = false;
};
int classify_host_views(const ikb_problem *p, int64_t B, const ikb_batch_io *io, HostViews *out);
// Stage the inputs of batch slice [b0, b1) on stream `s` (copy-in and, for compact targets, the SE3 expansion).
template <typename T> int stage_inputs(const ikb_problem *p, Staging<T> &st, const HostViews &hv, long long B, long long b0, long long b1,
                                       bool first, cudaStream_t s, bool expand = true);
// The SE3 expansion alone (expand = false above leaves it to the caller's compute stream).
template <typename T> int expand_staged(const ikb_problem *p, Staging<T> &st, const HostViews &hv, long long B, long long b0, long long b1,
                                        bool first, cudaStream_t s);
// Make sure the staging buffers of `st` hold a batch of B problems; fills the device view `dio` (pointers + dense strides).
template <typename T> int prepare_staging(const ikb_problem *p, Staging<T> &st, const HostViews &hv, long long B, ikb_batch_io *dio);
template <typename T> int ensure(T *&ptr, size_t &cap, size_t need) {
    if (need <= cap) return IKB_OK;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    size_t want = std::max(need, (size_t)1024);
    IKB_CUDA(cudaMalloc(&ptr, want * sizeof(T)));
    cap = want;
    return IKB_OK;
}

// ---- the solve launcher (ikb_solve.cu) ----
// Pipelined host path (solve_host): the inputs of batch slice [begin[c], begin[c + 1]) are on the device once `ready[c]`
// has happened.  The BULK launch is issued per slice, alternating between the caller's stream and `aux`, so that it
// overlaps the host-to-device copy of the next slices; the TAIL launch continues the stragglers of all slices at once.
struct ChunkPlan {
    int n = 0;
    long long begin[9] = {};
    cudaEvent_t ready[8] = {};
    cudaStream_t aux = nullptr;
    cudaEvent_t ev_aux = nullptr, ev_main = nullptr;
    // work that must precede slice c's launch on ITS compute stream (the SE3 expansion of compact targets: a kernel, which
    // in the copy stream would wait for the previous slice's persistent launch and hold the next slices' copies back)
    std::function<int(int, cudaStream_t)> pre;
};

// Merged launch of the pipelined queue (ikb_queue_*): `nseg` batches, each with its own buffers (host array of segment
// descriptors sorted by `begin`; launch_solve copies them into the kernel parameters).
template <typename T> struct Merged {
    const BatchSeg<T> *seg;
    int nseg;
};

// Is this solve going to take the two-launch (BULK + TAIL) path?  (the only one that can be pipelined by slices)
bool two_phase(const ikb_problem *p, const ikb_dls_params *prm, int64_t B, int *cap_out = nullptr);

// Enqueue ik::dls for B problems on stream `s`: picks the kernels (specialised BULK + TAIL pair, latency configuration,
// team kernel, generic kernel) and the scratch.  `io` holds DEVICE pointers (nullptr for a merged launch).
// Extra outputs of the *_solve_ex calls (device pointers, [B][nv] / [B][rows] / [B][rows][nv]); forces the table-driven kernel.
template <typename T> struct SolveAux {
    T *dq = nullptr, *e = nullptr, *J = nullptr;
};
template <typename T>
int launch_solve(const ikb_problem *p, const ikb_dls_params *prm, int64_t B, const ikb_batch_io *io, cudaStream_t s,
                 const ChunkPlan *plan = nullptr, const Merged<T> *merged = nullptr, const double *pik_lambda = nullptr,
                 const SolveAux<T> *aux = nullptr);
// (pik_lambda != nullptr: ik::pik instead of ik::dls -- per-level damping, table-driven kernel only)

// Carried stragglers (pipelined queue): a merged BULK launch whose stragglers have not been continued yet.  `tail` is
// the complete argument block of the TAIL launch that would finish them (resume = 1: suspended list, its count, the
// saved step counts, the group's segment table, the solver parameters); the NEXT merged launch of the queue continues
// them instead (launch_merged_carry), beside its own problems, and only a queue that runs empty launches the TAIL.
template <typename T> struct CarryState {
    bool valid = false;
    SolveArgs<T> tail;
};
// Queue-owned scratch of one merged launch (two sets, used alternately): suspended list, step counts, 4 counters.
struct CarryScratch {
    unsigned int *list = nullptr;
    int *iters = nullptr;
    unsigned long long *counters = nullptr;
    size_t cap = 0;
};
// BULK launch of a merged group that first continues `in`'s stragglers (in may be null / invalid); its own stragglers
// are left suspended and described by `out`.  Requires a specialised kernel and two_phase(p, prm, B).
template <typename T>
int launch_merged_carry(const ikb_problem *p, const ikb_dls_params *prm, int64_t B, const Merged<T> *merged, cudaStream_t s,
                        const CarryScratch &own, const CarryState<T> *in, CarryState<T> *out);
// The TAIL launch that finishes `c`'s stragglers.
template <typename T> int launch_carry_tail(const ikb_problem *p, const CarryState<T> &c, cudaStream_t s);

// Size class of the team-per-problem kernel: the problem's class, except that a class-2 problem (up to 30 rows) on a
// Cassie-sized tree takes the smaller scratch of CoopClass<3> (dls_coop.cuh).  IKB_COOP_CLASS3=0 disables it (A/B runs).
inline int coop_class(const ikb_problem *p) {
    const char *e = std::getenv("IKB_COOP_CLASS3");
    const HostModel &m = p->hp.model;
    if (p->size_class == 2 && m.njoints() <= 20 && m.nv <= 24 && m.nq <= 28 && !(e && e[0] == '0')) return 3;
    return p->size_class;
}

// The table-driven team-per-problem kernel (ikb_coop.cu / dls_coop.cuh) for size class `cls`.
template <typename T>
int launch_coop(int cls, const DevProblem<T> *dP, const SolveArgs<T> &a, bool pik, int extra /* 0 plain, 1 CoM, 2 constraints */, bool shfl, int sm_count,
                cudaStream_t s);

}  // namespace capi
}  // namespace ikb
