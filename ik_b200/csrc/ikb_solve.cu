// The solve launcher and the host-buffer path of the C ABI (include/ikb200.h): ikb_dls_solve_batch,
// ikb_dls_solve_batch_host, ikb_dls_solve.  The pipelined queue (ikb_queue.cu) launches through launch_solve too.
#include <cstdio>
#include <cstring>
#include <type_traits>

#include "capi_internal.hpp"
#include "dls_generic.cuh"

using namespace ikb;
using namespace ikb::capi;

namespace {

template <typename T> struct KernelTable {
    using Fn = void (*)(const DevProblem<T> *, SolveArgs<T>);
    static Fn dls(int cls) {
        switch (cls) {
            case 0: return dls_generic_kernel<T, 10, 8, 6>;
            case 1: return dls_generic_kernel<T, 20, 24, 12>;
            default: return dls_generic_kernel<T, 32, 36, 30>;
        }
    }
    static Fn pik(int cls) {  // ik::pik (pik.cpp:31-96)
        switch (cls) {
            case 0: return dls_generic_kernel<T, 10, 8, 6, true>;
            case 1: return dls_generic_kernel<T, 20, 24, 12, true>;
            default: return dls_generic_kernel<T, 32, 36, 30, true>;
        }
    }
};

// max_iterations <= 0: the reference returns q0 untouched, success = false, nothing evaluated
template <typename T> __global__ void passthrough_kernel(SolveArgs<T> a, int nq) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    for (int k = 0; k < nq; ++k) a.q[k * a.q_es + b * a.q_bs] = a.q0[k * a.q0_es + b * a.q0_bs];
    if (a.success) a.success[b] = 0;
    if (a.iters) a.iters[b] = 0;
    if (a.resid) a.resid[b] = T(0);
}

template <typename T> DevProblem<T> *dev_blob(const ikb_problem *p);
template <> DevProblem<double> *dev_blob<double>(const ikb_problem *p) { return p->d64; }
template <> DevProblem<float> *dev_blob<float>(const ikb_problem *p) { return p->d32; }

__global__ void set_ticket_kernel(unsigned long long *t, unsigned long long v) { *t = v; }

// One thread per problem: expand the compact record (quaternion / translation per FrameTask) to the SE3 record the
// kernels read.  Both arrays are dense, in the same orientation (strides passed in).
template <typename T>
__global__ void expand_targets_kernel(const __grid_constant__ ExpandTable tab, const T *__restrict__ c, long long c_es, long long c_bs,
                                      T *__restrict__ o, long long o_es, long long o_bs, long long b0, long long b1) {
    const long long b = b0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= b1) return;
    const T *cb = c + b * c_bs;
    T *ob = o + b * o_bs;
    for (int t = 0; t < tab.ntasks; ++t) {
        const T *ci = cb + tab.coff[t] * c_es;
        T *oi = ob + tab.toff[t] * o_es;
        const int mode = tab.mode[t];
        if (mode == 0) {
            for (int k = 0; k < tab.n[t]; ++k) oi[k * o_es] = ci[k * c_es];
            continue;
        }
        T R[9] = {T(1), T(0), T(0), T(0), T(1), T(0), T(0), T(0), T(1)}, tr[3] = {T(0), T(0), T(0)};
        if (mode == 1 || mode == 3) quat_to_rot(ci[0], ci[c_es], ci[2 * c_es], ci[3 * c_es], R);
        if (mode == 1) { tr[0] = ci[4 * c_es]; tr[1] = ci[5 * c_es]; tr[2] = ci[6 * c_es]; }
        if (mode == 2) { tr[0] = ci[0]; tr[1] = ci[c_es]; tr[2] = ci[2 * c_es]; }
        for (int k = 0; k < 9; ++k) oi[k * o_es] = R[k];
        for (int k = 0; k < 3; ++k) oi[(9 + k) * o_es] = tr[k];
    }
}
}  // namespace

namespace ikb {
namespace capi {

int check_solve_args(const ikb_problem *p, int dtype, const ikb_dls_params *prm, int64_t B, const ikb_batch_io *io) {
    if (!p || !prm || !io) return fail(IKB_ERR_INVALID_ARG, "null argument");
    if (!p->finalized) return fail(IKB_ERR_NOT_FINALIZED, "call ikb_problem_finalize first");
    if (dtype != IKB_F64 && dtype != IKB_F32) return fail(IKB_ERR_INVALID_ARG, "dtype must be IKB_F64 or IKB_F32");
    if (B < 0 || prm->max_iterations < 0) return fail(IKB_ERR_INVALID_ARG, "negative batch size or iteration count");
    if (B > 0 && (!io->q0 || !io->q || (!io->targets && p->hp.target_size() > 0)))
        return fail(IKB_ERR_INVALID_ARG, "q0, targets and q must be non-null");
    return IKB_OK;
}

constexpr int kCarryCapDefault = 1;   // step cap of a BULK launch whose stragglers are carried into the next one (measured: tools/carry_sweep.sh, profiles/r2_s3_carry_sweep.txt)

// Is this solve going to take the two-launch (BULK + TAIL) path?  (the only one that can be pipelined by slices)
bool two_phase(const ikb_problem *p, const ikb_dls_params *prm, int64_t B, int *cap_out) {
    const char *cap_env = std::getenv("IKB_BULK_CAP");
    const int cap = cap_env ? std::atoi(cap_env) : 16;
    if (cap_out) *cap_out = cap;
    return p->spec && B > 2LL * 32 * p->sm_count && cap > 0 && prm->max_iterations > cap;
}

// Scratch of a two-launch solve (suspended-problem list, step counts): slot `slot` of the problem's ring, grown to B
// entries; stream `s` waits for the slot's previous user.  The descriptor is COPIED out under the lock, and a buffer that
// is replaced by a larger one is retired (freed with the handle), never freed: another host thread may be about to launch
// with the old pointers, and launches already in flight keep using them.
static int acquire_scratch(const ikb_problem *p, unsigned slot, int64_t B, cudaStream_t s, SolveScratch *out) {
    ikb_problem *mp = const_cast<ikb_problem *>(p);
    std::lock_guard<std::mutex> lk(mp->scratch_mu);
    if (mp->scratch[0].cap < (size_t)B) {
        for (auto &x : mp->scratch) {
            if (x.list) mp->retired.push_back(x.list);
            if (x.iters) mp->retired.push_back(x.iters);
            x.list = nullptr; x.iters = nullptr; x.cap = 0;
            IKB_CUDA(cudaMalloc(&x.list, (size_t)B * sizeof(unsigned int)));
            IKB_CUDA(cudaMalloc(&x.iters, (size_t)B * sizeof(int)));
            x.cap = (size_t)B;
            if (!x.ev) IKB_CUDA(cudaEventCreateWithFlags(&x.ev, cudaEventDisableTiming));
        }
    }
    *out = mp->scratch[slot % kScratchSlots];
    IKB_CUDA(cudaStreamWaitEvent(s, out->ev, 0));  // the slot's previous user (any stream) must be done
    return IKB_OK;
}

template <typename T>
static int launch_solve_impl(const ikb_problem *p, const ikb_dls_params *prm, int64_t B, const ikb_batch_io *io, cudaStream_t s,
                             const ChunkPlan *plan, const Merged<T> *merged, const double *pik_lambda, const SolveAux<T> *aux,
                             unsigned slot) {
    SolveArgs<T> a{};
    if (!merged) {
        a.q0 = (const T *)io->q0; a.q0_es = io->q0_elem_stride; a.q0_bs = io->q0_batch_stride;
        a.targets = (const T *)io->targets; a.tg_es = io->targets_elem_stride; a.tg_bs = io->targets_batch_stride;
        a.q = (T *)io->q; a.q_es = io->q_elem_stride; a.q_bs = io->q_batch_stride;
        a.success = io->success;
        a.iters = io->iters;
        a.resid = (T *)io->resid;
        a.nseg = 0;
    } else {
        if (!p->spec || prm->max_iterations <= 0) return fail(IKB_ERR_INVALID_ARG, "internal: merged launch on a problem without a specialised kernel");
        a.nseg = merged->nseg;
        for (int i = 0; i < kMaxSegments; ++i) {
            if (i < merged->nseg) a.seg[i] = merged->seg[i];
            else a.seg[i].begin = LLONG_MAX;
        }
    }
    a.B = B;
    a.max_iterations = prm->max_iterations;
    a.step_length = (T)prm->step_length;
    a.damping2 = (T)(prm->damping * prm->damping);
    a.tolerance = (T)prm->tolerance;
    a.ticket = p->d_tickets + slot * 16;  // 128 B apart
    if (aux) { a.aux_dq = aux->dq; a.aux_e = aux->e; a.aux_J = aux->J; }
    IKB_CUDA(cudaMemsetAsync(a.ticket, 0, sizeof(unsigned long long), s));

    if (prm->max_iterations <= 0) {
        // dls.cpp:14 never enters the loop: q0 is returned with success = false (dls.cpp:76-77)
        const int threads = 128;
        passthrough_kernel<T><<<(unsigned)((B + threads - 1) / threads), threads, 0, s>>>(a, p->hp.model.nq);
        IKB_CUDA(cudaGetLastError());
        g_launches.fetch_add(1);
        return IKB_OK;
    }
    a.it_cap = INT_MAX;
    a.resume = 0;
    a.list = nullptr;
    a.list_count = nullptr;
    a.iters_ws = merged ? nullptr : io->iters;
    for (int l = 0; l < kPikMaxLevels; ++l) a.pik_lambda2[l] = pik_lambda ? (T)(pik_lambda[l] * pik_lambda[l]) : T(0);
    if (p->spec && !pik_lambda && !aux) {
        const SpecHostConsts hc{p->hp.model.lower.data(), p->hp.model.upper.data(), p->weight_stacked.data(), p->mask_stacked.data()};
        // Scheduling (DESIGN.md 4.1).  A batch that the latency configuration keeps resident in one wave runs there
        // directly.  A larger batch runs BULK (throughput configuration) with a step cap: the few problems still
        // unfinished after `cap` steps -- the reference lets them run to max_iterations, 100 by default -- are suspended
        // and a TAIL launch continues all of them at once, each group of 32 with an SM's schedulers to itself, instead
        // of letting them trickle out of the bulk kernel one 100-step straggler at a time.
        const long long wave = 2LL * 32 * p->sm_count;
        int cap;
        const bool two = two_phase(p, prm, B, &cap);
        int rc;
        if (plan && !two) return fail(IKB_ERR_INVALID_ARG, "internal: slice plan on a single-launch solve");
        if (B <= wave) {
            rc = launch_specialized<T>(*p->spec, hc, a, SPEC_TAIL, B, p->sm_count, s);
            if (rc == IKB_OK) g_launches.fetch_add(1);
        } else if (cap <= 0 || prm->max_iterations <= cap) {
            rc = launch_specialized<T>(*p->spec, hc, a, SPEC_BULK, B, p->sm_count, s);
            if (rc == IKB_OK) g_launches.fetch_add(1);
        } else {
            SolveScratch scv, *sc = &scv;
            if ((rc = acquire_scratch(p, slot, B, s, sc))) return rc;
            IKB_CUDA(cudaMemsetAsync(a.ticket, 0, 3 * sizeof(unsigned long long), s));  // bulk ticket, tail ticket, list count
            a.it_cap = cap;
            a.list = sc->list;
            a.list_count = a.ticket + 2;
            a.iters_ws = (!merged && io->iters) ? io->iters : sc->iters;
            if (!plan) {
                rc = launch_specialized<T>(*p->spec, hc, a, SPEC_BULK, B, p->sm_count, s);
                if (rc == IKB_OK) g_launches.fetch_add(1);
            } else {
                // one BULK launch per slice: its tickets run from begin[c] to begin[c + 1] (own counter, words 3.. of the slot)
                rc = IKB_OK;
                IKB_CUDA(cudaEventRecord(plan->ev_main, s));  // counters zeroed
                IKB_CUDA(cudaStreamWaitEvent(plan->aux, plan->ev_main, 0));
                for (int c = 0; c < plan->n && rc == IKB_OK; ++c) {
                    cudaStream_t cs = (c & 1) ? plan->aux : s;
                    IKB_CUDA(cudaStreamWaitEvent(cs, plan->ready[c], 0));
                    if (plan->pre && (rc = plan->pre(c, cs)) != IKB_OK) break;
                    SolveArgs<T> ac = a;
                    ac.ticket = a.ticket + 3 + c;
                    ac.B = plan->begin[c + 1];
                    set_ticket_kernel<<<1, 1, 0, cs>>>(ac.ticket, (unsigned long long)plan->begin[c]);
                    rc = launch_specialized<T>(*p->spec, hc, ac, SPEC_BULK, plan->begin[c + 1] - plan->begin[c], p->sm_count, cs);
                    if (rc == IKB_OK) g_launches.fetch_add(2);
                }
                IKB_CUDA(cudaEventRecord(plan->ev_aux, plan->aux));
                IKB_CUDA(cudaStreamWaitEvent(s, plan->ev_aux, 0));
            }
            if (rc == IKB_OK) {
                SolveArgs<T> t = a;
                t.resume = 1;
                t.it_cap = INT_MAX;
                t.ticket = a.ticket + 1;
                rc = launch_specialized<T>(*p->spec, hc, t, SPEC_TAIL, B, p->sm_count, s);
                if (rc == IKB_OK) g_launches.fetch_add(1);
            }
            IKB_CUDA(cudaEventRecord(sc->ev, s));
        }
        if (rc != IKB_OK) return cuda_fail(cudaGetLastError(), "specialised kernel launch");
        return IKB_OK;
    }
    if (merged) return fail(IKB_ERR_INVALID_ARG, "internal: merged launch on the table-driven kernel");
    // Table-driven problems: the team-per-problem kernel (dls_coop.cuh; J in shared memory, Gram rows and the factorisation
    // in registers).  IKB_GENERIC_LEGACY=1 keeps the thread-per-problem local-memory kernel (dls_generic.cuh) for A/B runs;
    // it is also the fallback for problems beyond the cooperative kernel's table capacities.
    const char *legacy_env = std::getenv("IKB_GENERIC_LEGACY");
    if (aux && !p->coop_ok) return fail(IKB_ERR_UNSUPPORTED, "dq / e / J outputs need the team-per-problem kernel (problem exceeds its table capacities)");
    if (p->coop_ok && (aux || !(legacy_env && legacy_env[0] == '1'))) {
        const char *shfl_env = std::getenv("IKB_COOP_SHFL");
        const bool shfl = shfl_env ? shfl_env[0] == '1' : false;   // measured: the shared-memory column is 3-8 % faster (DESIGN.md 4.2)
        int extra = p->hp.constraints.empty() ? 0 : 2;   // scratch level: 1 = CentreOfMassTask arrays, 2 = + projection buffers (and always ik::pik)
        for (const auto &t : p->hp.tasks)
            if (t.kind == IKB_TASK_COM && extra < 1) extra = 1;
        if (launch_coop<T>(coop_class(p), dev_blob<T>(p), a, pik_lambda != nullptr, extra, shfl, p->sm_count, s))
            return cuda_fail(cudaGetLastError(), "team-per-problem kernel launch");
        g_launches.fetch_add(1);
        return IKB_OK;
    }
    auto fn = pik_lambda ? KernelTable<T>::pik(p->size_class) : KernelTable<T>::dls(p->size_class);
    const char *thr_env = std::getenv("IKB_GENERIC_THREADS"), *bps_env = std::getenv("IKB_GENERIC_BLOCKS_PER_SM");
    const int threads = thr_env ? std::max(32, std::min(128, std::atoi(thr_env) / 32 * 32)) : 128;
    const size_t smem = sizeof(DevProblem<T>) + 16;
    int per_sm = 0;
    IKB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, smem));
    if (per_sm < 1) per_sm = 1;
    if (bps_env && std::atoi(bps_env) > 0) per_sm = std::min(per_sm, std::atoi(bps_env));
    long long blocks = (B + threads - 1) / threads;
    blocks = std::min<long long>(blocks, (long long)per_sm * p->sm_count);
    // Two launches for a batch that more than fills the GPU (DESIGN.md 4.2): problems unfinished after `cap` steps are
    // parked and a second launch continues them, 32 to a warp and one warp per CTA, so that a straggler's local-memory
    // scratch shares its cache lines with 31 others and stays in L1 instead of thrashing it from a mostly idle warp.
    const char *cap_env = std::getenv("IKB_GENERIC_CAP");
    const int cap = cap_env ? std::atoi(cap_env) : 32;  // measured: profiles/r1_generic_two_launch.txt (16 suits quick problems, 32 never loses to one launch)
    if (cap > 0 && prm->max_iterations > cap && B > 2048) {
        SolveScratch scv, *sc = &scv;
        int rc;
        if ((rc = acquire_scratch(p, slot, B, s, sc))) return rc;
        IKB_CUDA(cudaMemsetAsync(a.ticket, 0, 3 * sizeof(unsigned long long), s));  // first ticket, second ticket, list count
        a.it_cap = cap;
        a.list = sc->list;
        a.list_count = a.ticket + 2;
        a.iters_ws = io->iters ? io->iters : sc->iters;
        fn<<<(unsigned)blocks, threads, smem, s>>>(dev_blob<T>(p), a);
        IKB_CUDA(cudaGetLastError());
        SolveArgs<T> t = a;
        t.resume = 1;
        t.it_cap = INT_MAX;
        t.ticket = a.ticket + 1;
        int per_sm1 = 0;
        IKB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm1, fn, 32, smem));
        const long long blocks1 = std::min<long long>((B + 31) / 32, (long long)std::max(per_sm1, 1) * p->sm_count);
        fn<<<(unsigned)blocks1, 32, smem, s>>>(dev_blob<T>(p), t);
        IKB_CUDA(cudaGetLastError());
        IKB_CUDA(cudaEventRecord(sc->ev, s));
        g_launches.fetch_add(2);
        return IKB_OK;
    }
    fn<<<(unsigned)blocks, threads, smem, s>>>(dev_blob<T>(p), a);
    IKB_CUDA(cudaGetLastError());
    g_launches.fetch_add(1);
    return IKB_OK;
}

// The slot's ticket counters (and, for a two-launch solve, its scratch) are reused every kTicketSlots launches, possibly
// from another stream: stream `s` first waits for the event the slot's previous user recorded after its last kernel, and
// records its own when everything that reads the counters has been enqueued (ADVICE r1: the memset used to race with a
// long kernel of another stream).
template <typename T>
int launch_solve(const ikb_problem *p, const ikb_dls_params *prm, int64_t B, const ikb_batch_io *io, cudaStream_t s,
                 const ChunkPlan *plan, const Merged<T> *merged, const double *pik_lambda, const SolveAux<T> *aux) {
    const unsigned slot = const_cast<ikb_problem *>(p)->ticket_next.fetch_add(1) % kTicketSlots;
    IKB_CUDA(cudaStreamWaitEvent(s, p->ticket_ev[slot], 0));
    const int rc = launch_solve_impl<T>(p, prm, B, io, s, plan, merged, pik_lambda, aux, slot);
    IKB_CUDA(cudaEventRecord(p->ticket_ev[slot], s));
    return rc;
}

template <typename T>
int launch_merged_carry(const ikb_problem *p, const ikb_dls_params *prm, int64_t B, const Merged<T> *merged, cudaStream_t s,
                        const CarryScratch &own, const CarryState<T> *in, CarryState<T> *out) {
    int cap = 0;
    if (!p->spec || !merged || !two_phase(p, prm, B, &cap) || own.cap < (size_t)B)
        return fail(IKB_ERR_INVALID_ARG, "internal: carried launch needs a specialised two-launch solve and scratch for the group");
    // A carried launch hands its stragglers to the NEXT launch, where they run among fresh problems at the throughput
    // configuration's rate: suspending early costs nothing, and it cuts the end of this launch, where ever fewer slots are
    // busy, to a few trips.  (The TAIL launch of the two-launch schedule is latency-bound instead: there a late
    // hand-over, IKB_BULK_CAP = 16, keeps the list short.)  IKB_CARRY_CAP overrides the measured default.
    {
        const char *e = std::getenv("IKB_CARRY_CAP");
        const int ccap = e ? std::atoi(e) : kCarryCapDefault;
        if (ccap >= 1 && ccap < cap) cap = ccap;
    }
    SolveArgs<T> a{};
    a.nseg = merged->nseg;
    for (int i = 0; i < kMaxSegments; ++i) {
        if (i < merged->nseg) a.seg[i] = merged->seg[i];
        else a.seg[i].begin = LLONG_MAX;
        a.cseg[i].begin = LLONG_MAX;
    }
    a.B = B;
    a.max_iterations = prm->max_iterations;
    a.step_length = (T)prm->step_length;
    a.damping2 = (T)(prm->damping * prm->damping);
    a.tolerance = (T)prm->tolerance;
    a.ticket = own.counters;             // [0] bulk tickets, [1] tail tickets, [2] suspended count
    IKB_CUDA(cudaMemsetAsync(own.counters, 0, 4 * sizeof(unsigned long long), s));
    a.it_cap = cap;
    a.resume = 0;
    a.list = own.list;
    a.list_count = own.counters + 2;
    a.iters_ws = own.iters;
    if (in && in->valid) {
        a.carry_list = in->tail.list;
        a.carry_count = in->tail.list_count;
        a.carry_iters = in->tail.iters_ws;
        for (int i = 0; i < kMaxSegments; ++i) a.cseg[i] = in->tail.seg[i];
    }
    const SpecHostConsts hc{p->hp.model.lower.data(), p->hp.model.upper.data(), p->weight_stacked.data(), p->mask_stacked.data()};
    if (launch_specialized<T>(*p->spec, hc, a, SPEC_BULK, B, p->sm_count, s) != IKB_OK) return cuda_fail(cudaGetLastError(), "specialised kernel launch");
    g_launches.fetch_add(1);
    out->valid = true;
    out->tail = a;
    out->tail.resume = 1;
    out->tail.it_cap = INT_MAX;
    out->tail.ticket = own.counters + 1;
    out->tail.carry_list = nullptr;
    out->tail.carry_count = nullptr;
    out->tail.carry_iters = nullptr;
    return IKB_OK;
}
template <typename T> int launch_carry_tail(const ikb_problem *p, const CarryState<T> &c, cudaStream_t s) {
    if (!c.valid) return IKB_OK;
    const SpecHostConsts hc{p->hp.model.lower.data(), p->hp.model.upper.data(), p->weight_stacked.data(), p->mask_stacked.data()};
    if (launch_specialized<T>(*p->spec, hc, c.tail, SPEC_TAIL, c.tail.B, p->sm_count, s) != IKB_OK) return cuda_fail(cudaGetLastError(), "specialised kernel launch");
    g_launches.fetch_add(1);
    return IKB_OK;
}
template int launch_merged_carry<double>(const ikb_problem *, const ikb_dls_params *, int64_t, const Merged<double> *, cudaStream_t, const CarryScratch &,
                                         const CarryState<double> *, CarryState<double> *);
template int launch_merged_carry<float>(const ikb_problem *, const ikb_dls_params *, int64_t, const Merged<float> *, cudaStream_t, const CarryScratch &,
                                        const CarryState<float> *, CarryState<float> *);
template int launch_carry_tail<double>(const ikb_problem *, const CarryState<double> &, cudaStream_t);
template int launch_carry_tail<float>(const ikb_problem *, const CarryState<float> &, cudaStream_t);

template int launch_solve<double>(const ikb_problem *, const ikb_dls_params *, int64_t, const ikb_batch_io *, cudaStream_t,
                                  const ChunkPlan *, const Merged<double> *, const double *, const SolveAux<double> *);
template int launch_solve<float>(const ikb_problem *, const ikb_dls_params *, int64_t, const ikb_batch_io *, cudaStream_t,
                                 const ChunkPlan *, const Merged<float> *, const double *, const SolveAux<float> *);

// ---- host views, staging, compact targets ----------------------------------------------------------------------------
int classify_host_views(const ikb_problem *p, int64_t B, const ikb_batch_io *io, HostViews *out) {
    const int nq = p->hp.model.nq;
    out->compact = io->targets_format == IKB_TARGETS_COMPACT;
    if (io->targets_format != IKB_TARGETS_SE3 && io->targets_format != IKB_TARGETS_COMPACT)
        return fail(IKB_ERR_INVALID_ARG, "targets_format must be IKB_TARGETS_SE3 or IKB_TARGETS_COMPACT (zero-initialise ikb_batch_io)");
    const int tsz = out->compact ? p->expand.csz : p->hp.target_size();
    out->q0 = host_view(io->q0, io->q0_elem_stride, io->q0_batch_stride, nq, B, true);
    out->tg = host_view(io->targets, io->targets_elem_stride, io->targets_batch_stride, tsz, B, true);
    out->q = host_view(io->q, io->q_elem_stride, io->q_batch_stride, nq, B, false);
    if (out->q0.kind == VIEW_BAD || out->tg.kind == VIEW_BAD || out->q.kind == VIEW_BAD)
        return fail(IKB_ERR_INVALID_ARG, "host views must be SoA rows (batch_stride 1, elem_stride >= B), AoS records (elem_stride 1, "
                                         "batch_stride >= element count) or, for inputs, a broadcast (batch_stride 0)");
    return IKB_OK;
}

template <typename T>
int prepare_staging(const ikb_problem *p, Staging<T> &st, const HostViews &hv, long long B, ikb_batch_io *dio) {
    const int tsz = p->hp.target_size();
    int rc;
    // the SE3 targets the kernels read: as copied in, or expanded from the compact record in the same orientation
    HostView tgd = hv.tg;
    tgd.n = tsz;
    if ((rc = ensure(st.q0, st.q0_cap, std::max<size_t>(hv.q0.dev_count(B), 1))) || (rc = ensure(st.targets, st.tg_cap, std::max<size_t>(tgd.dev_count(B), 1))) ||
        (rc = ensure(st.q, st.q_cap, std::max<size_t>(hv.q.dev_count(B), 1))) || (rc = ensure(st.resid, st.b_cap, (size_t)std::max<long long>(B, 1))))
        return rc;
    if (hv.compact && (rc = ensure(st.compact, st.compact_cap, std::max<size_t>(hv.tg.dev_count(B), 1)))) return rc;
    dio->q0 = st.q0; dio->q0_elem_stride = hv.q0.dev_es(B); dio->q0_batch_stride = hv.q0.dev_bs();
    dio->targets = st.targets; dio->targets_elem_stride = tgd.dev_es(B); dio->targets_batch_stride = tgd.dev_bs();
    dio->q = st.q; dio->q_elem_stride = hv.q.dev_es(B); dio->q_batch_stride = hv.q.dev_bs();
    dio->resid = st.resid;
    dio->targets_format = IKB_TARGETS_SE3;
    return IKB_OK;
}

template <typename T>
int stage_inputs(const ikb_problem *p, Staging<T> &st, const HostViews &hv, long long B, long long b0, long long b1, bool first, cudaStream_t s,
                 bool expand) {
    int rc;
    if ((rc = copy_view_in<T>(st.q0, hv.q0, B, b0, b1, first, s))) return rc;
    if (!hv.compact) return copy_view_in<T>(st.targets, hv.tg, B, b0, b1, first, s);
    if ((rc = copy_view_in<T>(st.compact, hv.tg, B, b0, b1, first, s))) return rc;
    if (!expand) return IKB_OK;   // the caller runs expand_staged on its compute stream
    return expand_staged<T>(p, st, hv, B, b0, b1, first, s);
}

// Compact targets -> SE3 records on the device (one thread per problem).  A KERNEL: in a copy stream it would sit behind a
// persistent solve kernel that holds every SM's registers, and the stream's later copies behind it (ikb_queue.cu).
template <typename T>
int expand_staged(const ikb_problem *p, Staging<T> &st, const HostViews &hv, long long B, long long b0, long long b1, bool first, cudaStream_t s) {
    if (!hv.compact) return IKB_OK;
    // a broadcast compact record expands to one broadcast SE3 record (one "problem")
    const bool bc = hv.tg.kind == VIEW_BCAST;
    if (bc && !first) return IKB_OK;
    const long long e0 = bc ? 0 : b0, e1 = bc ? 1 : b1;
    if (e1 <= e0) return IKB_OK;
    HostView tgd = hv.tg;
    tgd.n = p->hp.target_size();
    const int threads = 128;
    expand_targets_kernel<T><<<(unsigned)((e1 - e0 + threads - 1) / threads), threads, 0, s>>>(
        p->expand, st.compact, hv.tg.dev_es(B), hv.tg.dev_bs(), st.targets, tgd.dev_es(B), tgd.dev_bs(), e0, e1);
    IKB_CUDA(cudaGetLastError());
    g_launches.fetch_add(1);
    return IKB_OK;
}
template int prepare_staging<double>(const ikb_problem *, Staging<double> &, const HostViews &, long long, ikb_batch_io *);
template int prepare_staging<float>(const ikb_problem *, Staging<float> &, const HostViews &, long long, ikb_batch_io *);
template int stage_inputs<double>(const ikb_problem *, Staging<double> &, const HostViews &, long long, long long, long long, bool, cudaStream_t, bool);
template int stage_inputs<float>(const ikb_problem *, Staging<float> &, const HostViews &, long long, long long, long long, bool, cudaStream_t, bool);
template int expand_staged<double>(const ikb_problem *, Staging<double> &, const HostViews &, long long, long long, long long, bool, cudaStream_t);
template int expand_staged<float>(const ikb_problem *, Staging<float> &, const HostViews &, long long, long long, long long, bool, cudaStream_t);

}  // namespace capi
}  // namespace ikb

namespace {
template <typename T> Staging<T> &staging(ikb_problem *p);
template <> Staging<double> &staging<double>(ikb_problem *p) { return p->st64; }
template <> Staging<float> &staging<float>(ikb_problem *p) { return p->st32; }

// IKB_HOST_TRACE=1: print the device-side timeline of one host-path solve (debug aid for the e2e numbers in DESIGN.md)
struct HostTrace {
    bool on = false;
    std::vector<std::pair<const char *, cudaEvent_t>> ev;
    HostTrace() { const char *e = std::getenv("IKB_HOST_TRACE"); on = e && e[0] == '1'; }
    void mark(const char *name, cudaStream_t s) {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        ev.emplace_back(name, e);
    }
    void dump() {
        if (!on || ev.empty()) return;
        for (auto &x : ev) {
            float ms = 0;
            cudaEventSynchronize(x.second);
            cudaEventElapsedTime(&ms, ev[0].second, x.second);
            std::fprintf(stderr, "[ikb host trace] %-14s %8.3f ms\n", x.first, ms);
            }
        for (auto &x : ev) cudaEventDestroy(x.second);
        ev.clear();
    }
};

template <typename T>
int solve_host(ikb_problem *p, const ikb_dls_params *prm, int64_t B, const ikb_batch_io *io, const double *pik_lambda = nullptr,
               double *aux_dq = nullptr, double *aux_e = nullptr, double *aux_J = nullptr) {
    Staging<T> &st = staging<T>(p);
    HostViews hv;
    int rc;
    if ((rc = classify_host_views(p, B, io, &hv))) return rc;
    ikb_batch_io dio = *io;
    if ((rc = prepare_staging<T>(p, st, hv, B, &dio))) return rc;
    if ((size_t)B > p->st_flag_cap) {
        if (p->st_success) cudaFree(p->st_success);
        if (p->st_iters) cudaFree(p->st_iters);
        p->st_success = nullptr; p->st_iters = nullptr; p->st_flag_cap = 0;
        IKB_CUDA(cudaMalloc(&p->st_success, (size_t)B));
        IKB_CUDA(cudaMalloc(&p->st_iters, (size_t)B * sizeof(int)));
        p->st_flag_cap = (size_t)B;
    }
    cudaStream_t s = p->stream;
    HostTrace tr;
    tr.mark("start", s);
    dio.success = p->st_success;
    dio.iters = p->st_iters;
    // extra outputs of the *_solve_ex calls (FP64, tiny batches): device scratch freed right after the call
    SolveAux<T> aux;
    const int nv = p->hp.model.nv, rows = p->hp.rows();
    const bool want_aux = aux_dq || aux_e || aux_J;
    if (want_aux) {   // one buffer owned by the handle (a cudaMalloc per call would dominate a single solve)
        const size_t need = (size_t)B * ((size_t)nv + rows + (size_t)rows * nv) * sizeof(T);
        if (need > p->st_aux_cap) {
            if (p->st_aux) cudaFree(p->st_aux);
            p->st_aux = nullptr; p->st_aux_cap = 0;
            IKB_CUDA(cudaMalloc(&p->st_aux, need));
            p->st_aux_cap = need;
        }
        aux.dq = (T *)p->st_aux;
        aux.e = aux.dq + (size_t)B * nv;
        aux.J = aux.e + (size_t)B * rows;
    }
    // A two-launch solve is pipelined by batch slices: slice c + 1 crosses PCIe while the BULK launch of slice c runs
    // (the staging buffers are dense, so a slice is a 2-D or a contiguous copy).
    const char *slices_env = std::getenv("IKB_HOST_SLICES");
    const int nslice = (int)std::min<int64_t>(slices_env ? std::max(1, std::min(8, std::atoi(slices_env))) : 4, B / 8192);
    const char *pipe_env = std::getenv("IKB_HOST_PIPELINE");
    // (worth it only when the copy-in is long: the lean wire format -- compact targets, one shared q0: 6.8 MB for 65 536 Cassie
    // problems -- takes 1.17 ms unsliced against 1.26 ms in four slices, each with its own BULK launch; tools/blocking_compact.py)
    const double in_bytes = (double)sizeof(T) * (double)B *
                            ((hv.q0.kind == VIEW_BCAST ? 0.0 : (double)hv.q0.n) + (hv.tg.kind == VIEW_BCAST ? 0.0 : (double)hv.tg.n));
    const bool long_copy = slices_env || in_bytes >= 16e6;
    if (!pik_lambda && !want_aux && two_phase(p, prm, B) && nslice >= 2 && long_copy && !(pipe_env && pipe_env[0] == '0')) {
        ChunkPlan plan;
        plan.n = nslice;
        plan.aux = p->stream_aux;
        plan.ev_aux = p->ev_aux;
        plan.ev_main = p->ev_main;
        for (int c = 0; c <= nslice; ++c) plan.begin[c] = c == nslice ? B : (B / nslice * c) / 32 * 32;
        // the staging buffers may still be read by the previous call's kernels on `s`: order the copy stream behind it
        IKB_CUDA(cudaEventRecord(p->ev_main, s));
        IKB_CUDA(cudaStreamWaitEvent(p->stream_in, p->ev_main, 0));
        if (hv.compact)
            plan.pre = [&, p](int c, cudaStream_t cs) { return expand_staged<T>(p, st, hv, B, plan.begin[c], plan.begin[c + 1], c == 0, cs); };
        for (int c = 0; c < nslice; ++c) {
            if ((rc = stage_inputs<T>(p, st, hv, B, plan.begin[c], plan.begin[c + 1], c == 0, p->stream_in, false))) return rc;
            plan.ready[c] = p->ev_in[c];
            IKB_CUDA(cudaEventRecord(plan.ready[c], p->stream_in));
            tr.mark("h2d slice", p->stream_in);
        }
        if ((rc = launch_solve<T>(p, prm, B, &dio, s, &plan))) return rc;
    } else {
        if ((rc = stage_inputs<T>(p, st, hv, B, 0, B, true, s))) return rc;
        tr.mark("h2d", s);
        if ((rc = launch_solve<T>(p, prm, B, &dio, s, nullptr, nullptr, pik_lambda, want_aux ? &aux : nullptr))) return rc;
    }
    tr.mark("solve", s);
    if ((rc = copy_view_out<T>(hv.q, st.q, B, s))) return rc;
    if (io->success) IKB_CUDA(cudaMemcpyAsync(io->success, p->st_success, (size_t)B, cudaMemcpyDeviceToHost, s));
    if (io->iters) IKB_CUDA(cudaMemcpyAsync(io->iters, p->st_iters, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (io->resid) IKB_CUDA(cudaMemcpyAsync(io->resid, st.resid, (size_t)B * sizeof(T), cudaMemcpyDeviceToHost, s));
    if constexpr (std::is_same<T, double>::value) {
        if (aux_dq) IKB_CUDA(cudaMemcpyAsync(aux_dq, aux.dq, (size_t)B * nv * sizeof(T), cudaMemcpyDeviceToHost, s));
        if (aux_e) IKB_CUDA(cudaMemcpyAsync(aux_e, aux.e, (size_t)B * rows * sizeof(T), cudaMemcpyDeviceToHost, s));
        if (aux_J) IKB_CUDA(cudaMemcpyAsync(aux_J, aux.J, (size_t)B * rows * nv * sizeof(T), cudaMemcpyDeviceToHost, s));
    }
    tr.mark("d2h", s);
    IKB_CUDA(cudaStreamSynchronize(s));
    tr.dump();
    return IKB_OK;
}
}  // namespace

extern "C" {

int ikb_dls_solve_batch(const ikb_problem *p, int dtype, const ikb_dls_params *prm, int64_t B, const ikb_batch_io *io,
                        void *cuda_stream) {
    int rc = check_solve_args(p, dtype, prm, B, io);
    if (rc) return rc;
    if (B == 0) return IKB_OK;
    if (io->targets_format != IKB_TARGETS_SE3) return fail(IKB_ERR_INVALID_ARG, "compact targets are a wire format of the HOST entry points");
    DeviceGuard g(p->device);
    cudaStream_t s = (cudaStream_t)cuda_stream;
    return dtype == IKB_F64 ? launch_solve<double>(p, prm, B, io, s) : launch_solve<float>(p, prm, B, io, s);
}

int ikb_dls_solve_batch_host(ikb_problem *p, int dtype, const ikb_dls_params *prm, int64_t B, const ikb_batch_io *io) {
    int rc = check_solve_args(p, dtype, prm, B, io);
    if (rc) return rc;
    if (B == 0) return IKB_OK;
    DeviceGuard g(p->device);
    return dtype == IKB_F64 ? solve_host<double>(p, prm, B, io) : solve_host<float>(p, prm, B, io);
}

/* ---- ik::pik ---- */
void ikb_pik_params_default(ikb_pik_params *p) {
    if (!p) return;
    p->max_iterations = 100;  // pik.hpp:14
    p->step_length = 1.0;     // pik.hpp:16
    p->tolerance = 1e-4;      // visitor.hpp:19
    for (double &l : p->lambda) l = 1.0;  // pik_data::lambda (pik.hpp:31)
}

static int pik_to_dls(const ikb_problem *p, const ikb_pik_params *prm, ikb_dls_params *out) {
    if (!p || !prm) return fail(IKB_ERR_INVALID_ARG, "null argument");
    // the kernels hold kPikMaxLevels levels (DevProblem::level_rows, SolveArgs::pik_lambda2); max_priority_level itself
    // may be larger as long as no task sits above the table
    if (p->hp.levels() > kPikMaxLevels)
        return fail(IKB_ERR_UNSUPPORTED, "ik::pik holds at most 7 priority levels (ikb_pik_params::lambda): a task has priority above 6");
    ikb_dls_params_default(out);
    out->max_iterations = prm->max_iterations;
    out->step_length = prm->step_length;
    out->tolerance = prm->tolerance;
    return IKB_OK;
}

int ikb_pik_solve_batch(const ikb_problem *p, int dtype, const ikb_pik_params *prm, int64_t B, const ikb_batch_io *io, void *cuda_stream) {
    ikb_dls_params d;
    int rc = pik_to_dls(p, prm, &d);
    if (rc || (rc = check_solve_args(p, dtype, &d, B, io))) return rc;
    if (B == 0) return IKB_OK;
    if (io->targets_format != IKB_TARGETS_SE3) return fail(IKB_ERR_INVALID_ARG, "compact targets are a wire format of the HOST entry points");
    DeviceGuard g(p->device);
    cudaStream_t s = (cudaStream_t)cuda_stream;
    return dtype == IKB_F64 ? launch_solve<double>(p, &d, B, io, s, nullptr, nullptr, prm->lambda)
                            : launch_solve<float>(p, &d, B, io, s, nullptr, nullptr, prm->lambda);
}

int ikb_pik_solve_batch_host(ikb_problem *p, int dtype, const ikb_pik_params *prm, int64_t B, const ikb_batch_io *io) {
    ikb_dls_params d;
    int rc = pik_to_dls(p, prm, &d);
    if (rc || (rc = check_solve_args(p, dtype, &d, B, io))) return rc;
    if (B == 0) return IKB_OK;
    DeviceGuard g(p->device);
    return dtype == IKB_F64 ? solve_host<double>(p, &d, B, io, prm->lambda) : solve_host<float>(p, &d, B, io, prm->lambda);
}

static int solve_one(ikb_problem *p, const ikb_dls_params *prm, const double *pik_lambda, const double *q0, const double *targets,
                     double *q_out, int *success, int *iters, double *resid, double *dq, double *e, double *J) {
    const int nq = p->hp.model.nq, tsz = p->hp.target_size();
    uint8_t ok = 0;
    int32_t it = 0;
    double r = 0;
    ikb_batch_io io = {};
    io.q0 = q0; io.q0_elem_stride = 1; io.q0_batch_stride = nq;
    io.targets = targets; io.targets_elem_stride = 1; io.targets_batch_stride = tsz;
    io.q = q_out; io.q_elem_stride = 1; io.q_batch_stride = nq;
    io.success = &ok; io.iters = &it; io.resid = &r;
    int rc = check_solve_args(p, IKB_F64, prm, 1, &io);
    if (rc) return rc;
    DeviceGuard g(p->device);
    if ((rc = solve_host<double>(p, prm, 1, &io, pik_lambda, dq, e, J))) return rc;
    if (success) *success = ok;
    if (iters) *iters = it;
    if (resid) *resid = r;
    return IKB_OK;
}

int ikb_dls_solve(ikb_problem *p, const ikb_dls_params *prm, const double *q0, const double *targets, double *q_out,
                  int *success, int *iters, double *resid) {
    return ikb_dls_solve_ex(p, prm, q0, targets, q_out, success, iters, resid, nullptr, nullptr, nullptr);
}

int ikb_dls_solve_ex(ikb_problem *p, const ikb_dls_params *prm, const double *q0, const double *targets, double *q_out,
                     int *success, int *iters, double *resid, double *dq, double *e, double *J) {
    if (!p) return fail(IKB_ERR_INVALID_ARG, "null problem");
    ikb_dls_params dflt;
    ikb_dls_params_default(&dflt);
    return solve_one(p, prm ? prm : &dflt, nullptr, q0, targets, q_out, success, iters, resid, dq, e, J);
}

int ikb_pik_solve_ex(ikb_problem *p, const ikb_pik_params *prm, const double *q0, const double *targets, double *q_out,
                     int *success, int *iters, double *resid, double *dq, double *e, double *J) {
    ikb_pik_params dflt;
    ikb_pik_params_default(&dflt);
    if (!prm) prm = &dflt;
    ikb_dls_params d;
    int rc = pik_to_dls(p, prm, &d);
    if (rc) return rc;
    return solve_one(p, &d, prm->lambda, q0, targets, q_out, success, iters, resid, dq, e, J);
}

}  // extern "C"
