// Topology-specialised batched DLS IK kernel: the fast path of ikb_dls_solve_batch.
//
// The whole ik::dls loop (reference dls.cpp:14-74) runs in-kernel; its body is straight-line code generated for one
// fixed (tree, task list) pair by tools/gen_kernel.py (see its header for the arithmetic), so there are no tables, no
// dynamic indexing and no local memory.  Work decomposition:
//
//   * a GROUP of NWARPS warps owns 32 problem slots; lane l of every warp of the group works on slot l.  The warps
//     have ROLES (MPMD, no divergence: different warps may run different code): role k evaluates the tasks the
//     generator assigned to it -- FK of their supporting joints, SE3-log errors, weighted Jacobian non-zeros -- while
//     the other roles do theirs (Cassie: pelvis pose | left foot | right foot).  Role SOLVER then runs the fused
//     Gram + blocked LDL^T + substitutions and the step dq = -J^T y; every role integrates its own register copy of q
//     (bit-identical, same code and inputs), so no role ever waits for q.  Two named barriers per iteration
//     (bar.sync id, NWARPS*32): after evaluate (J, e visible) and after solve (dq, ||e||^2 visible).  Large systems
//     (Spec::PSOLVE, the humanoid) run the factorisation on all roles (Spec::psolve takes the group barrier as an
//     argument) and, with Spec::DSTEP, every role steps and writes the coordinates of q its own evaluate reads.
//   * per-problem state lives in strips of shared memory (element k of slot s at base[k * SLOTS + s]:
//     conflict-free): weighted J non-zeros, the LDL^T factor (whose storage first carries e and finally dq), the
//     target poses; plus ||e||^2 and a prefetched ticket per slot.  Cassie FP64: 219 doubles + 16 B = 1768 B per
//     problem -> 128 problems (4 groups, 12 warps) fill the 227 KB of an SM.
//   * limits and task weights arrive as a __grid_constant__ parameter, i.e. as constant-bank operands.
//
// Scheduling: persistent CTAs, one per SM; every SLOT pulls problem indices from a global ticket counter and refills
// itself the moment its problem converges or runs out of iterations, so all lanes execute the same body on every trip
// although iteration counts differ wildly across problems (median 4, p95 15, max 100 on the Cassie workload).  The
// SOLVER role knows ||e||^2 before everybody else and pulls the slot's next ticket right then (only if the slot is
// about to finish), so a refill costs no extra barrier and the atomic's latency hides behind the solve.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <type_traits>

#include "dev_problem.hpp"
#include "model.hpp"
#include "spec_common.hpp"
#include "specialized.hpp"
#include "tmem_scratch.cuh"

// 1: FP64 arrow kernels park the configuration registers in tensor memory between evaluate and step (tmem_scratch.cuh)
#ifndef IKB_TMEM_Q
#define IKB_TMEM_Q 1
#endif

namespace ikb {

constexpr int kSmemPerCtaMax = 227 * 1024;  // B200: 228 KB per SM, 227 KB usable by one CTA

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device (per-context) attribute: a process that finalizes problems
// on several GPUs must opt in on each of them.  One bit per device ordinal, set after the first successful call on
// that device (safe from concurrent host threads: a lost race only repeats the idempotent call).
struct DynSmemOptIn {
    std::atomic<unsigned long long> done{0};
    template <class Fn> bool ensure(Fn fn, int bytes) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return false;
        const unsigned long long bit = 1ULL << (dev & 63);
        if (done.load(std::memory_order_acquire) & bit) return true;
        if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess) return false;
        done.fetch_or(bit, std::memory_order_release);
        return true;
    }
};

// 1: arrow kernels stage a converged slot's next problem one trip ahead (kPrefetch below); 0 for A/B builds
#ifndef IKB_PREFETCH
#define IKB_PREFETCH 1
#endif

// Does the FP64 kernel of this spec keep the Jacobian strip in tensor memory?  (IKB_TMEM_J=0: never)
#ifndef IKB_TMEM_J
#define IKB_TMEM_J 1
#endif
template <class Spec, typename T> constexpr bool spec_tmem_j() { return IKB_TMEM_J && IKB_TMEM_Q && Spec::ARROW && Spec::TMEMJ && sizeof(T) == 8 && Spec::NQL <= 16; }
// Spec::qstage_l(role) (TMEMJ specs only): first of NQ factor-strip slots where a converged slot's next configuration is
// staged for that role; does every role of the spec have such a home?
template <class Spec, class = void> struct spec_qstage_l { static constexpr bool value = false; };
template <class Spec> struct spec_qstage_l<Spec, std::void_t<decltype(Spec::qstage_l(0))>> {
    static constexpr bool all(int r) { return r >= Spec::NWARPS || (Spec::qstage_l(r) >= 0 && all(r + 1)); }
    static constexpr bool value = all(0);
};

// IKB_TRIP_PROFILE=1 (tools/trip_profile.py; never in the library): the merged launch of a TMEMJ body adds up, per warp role,
// the clock64() cycles of each segment of a trip into ikb_trip_cycles (kTripSegs counters per role, then the trip count)
#ifndef IKB_TRIP_PROFILE
#define IKB_TRIP_PROFILE 0
#endif
enum TripSeg { kTripTopBarrier, kTripTmemFetch, kTripEvaluate, kTripPhase1, kTripStopTest, kTripPhase23, kTripBarrier2,
               kTripStep, kTripResults, kTripRefill, kTripPark, kTripSegs };
#if IKB_TRIP_PROFILE
static __device__ unsigned long long ikb_trip_cycles[4 * (kTripSegs + 1)];
#endif
struct TripClock {
#if IKB_TRIP_PROFILE
    long long t = 0, acc[kTripSegs] = {}, trips = 0;
    __device__ void start() { t = clock64(); }
    __device__ void trip() { ++trips; }
    __device__ void mark(int seg) {
        const long long now = clock64();
        acc[seg] += now - t;
        t = now;
    }
    // the results / refill split of the end of a trip: lanes run it divergently, so the warp's split point is the first
    // lane's `at` (0: this lane did not finish)
    __device__ void split(long long at) {
        unsigned d = at ? (unsigned)(at - t) : 0xffffffffu;
        d = __reduce_min_sync(0xffffffffu, d);
        if (d != 0xffffffffu) {
            acc[kTripResults] += d;
            t += d;
        }
        mark(kTripRefill);
    }
    __device__ void flush(int role) {
        if ((threadIdx.x & 31) != 0) return;
        for (int k = 0; k < kTripSegs; ++k) atomicAdd(&ikb_trip_cycles[role * (kTripSegs + 1) + k], (unsigned long long)acc[k]);
        atomicAdd(&ikb_trip_cycles[role * (kTripSegs + 1) + kTripSegs], (unsigned long long)trips);
    }
#else
    __device__ void start() {}
    __device__ void trip() {}
    __device__ void mark(int) {}
    __device__ void split(long long) {}
    __device__ void flush(int) {}
#endif
};
// tensor-memory columns of a warp role: 32 for the parked configuration + two per Jacobian slot of the role
template <class Spec, typename T> constexpr int spec_tmem_width(int role) { return 32 + (spec_tmem_j<Spec, T>() ? 2 * Spec::j_count(role) : 0); }
// columns in use in lane quarter `quarter` when the CTA has `nwarps` warps (warp w: quarter w % 4, role w % NWARPS)
template <class Spec, typename T> constexpr int spec_tmem_quarter(int quarter, int nwarps) {
    int c = 0;
    for (int w = quarter; w < nwarps; w += 4) c += spec_tmem_width<Spec, T>(w % Spec::NWARPS);
    return c;
}
template <class Spec, typename T> constexpr int spec_tmem_cols(int nwarps) {
    int m = 0;
    for (int qd = 0; qd < 4; ++qd) m = spec_tmem_quarter<Spec, T>(qd, nwarps) > m ? spec_tmem_quarter<Spec, T>(qd, nwarps) : m;
    return m <= 32 ? 32 : m <= 64 ? 64 : m <= 128 ? 128 : m <= 256 ? 256 : 512;
}

// (ik_b200/specialise.py spec_launch restates this to refuse, in words, a plugin spec that does not fit)
template <class Spec, typename T> struct SpecLaunch {
    static constexpr int NW = Spec::NWARPS;
    static constexpr bool kTmemJ = spec_tmem_j<Spec, T>();
    static constexpr int kStrip = (kTmemJ ? 0 : Spec::NSLOT) + Spec::NFACT + Spec::TSZ + 1;   // scalars per problem (+ ||e||^2)
    static constexpr int kBytesPerProblem = kStrip * (int)sizeof(T) + (int)sizeof(long long);  // + prefetched ticket
    static constexpr int kBySmem = kSmemPerCtaMax / (32 * kBytesPerProblem);               // groups that fit
    // register budget: 168 per thread for double, 128 for float -> at most 384 / 512 threads per (single) CTA
    static constexpr int kMaxThreads = sizeof(T) == 8 ? 384 : 512;
    static constexpr int kByRegs = kMaxThreads / (32 * NW);
    static constexpr int kG0 = kBySmem < kByRegs ? kBySmem : kByRegs;
    static constexpr int GROUPS = kG0 > 15 ? 15 : kG0;  // one named barrier per group (ids 1..15)
    static constexpr bool kFits = GROUPS >= 1;
    static constexpr int smem_bytes(int groups) { return groups * 32 * kBytesPerProblem; }
};

// SEG: merged launch of the pipelined queue (several batches, each with its own buffers: SolveArgs::seg).
template <class Spec, typename T, int GROUPS, int MINB, bool SEG>
__global__ void __launch_bounds__(GROUPS *Spec::NWARPS * 32, MINB)
    dls_spec_kernel(const __grid_constant__ SpecConsts<T, Spec::NQ, Spec::M> c, const __grid_constant__ SolveArgs<T> a) {
    constexpr int NQ = Spec::NQ, NV = Spec::NV, M = Spec::M, NW = Spec::NWARPS, SLOTS = GROUPS * 32;
    static_assert(Spec::NFACT >= M + NQ, "factor strip must also hold e and the stepped q");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int group = warp / NW, role = warp % NW;
    const int slot = group * 32 + lane;
    T *sm = reinterpret_cast<T *>(smem_raw) + slot;
    using S = Strip<T, SLOTS>;
    constexpr bool kTmemJ = spec_tmem_j<Spec, T>();         // the Jacobian strip lives in tensor memory, not here
    constexpr int kJS = kTmemJ ? 0 : Spec::NSLOT;
    const S sL{sm + kJS * SLOTS};                           // LDL^T factor
    const S sE{sm + (kJS + Spec::EOFF) * SLOTS};            //   ... M of whose slots carry e until the solve starts
    const S sD{sm + (kJS + M) * SLOTS};                     //   ... and whose next NQ slots carry the stepped q after it
    const S sT{sm + (kJS + Spec::NFACT) * SLOTS};           // target poses
    T *sRes = sm + (kJS + Spec::NFACT + Spec::TSZ) * SLOTS;  // ||e[0]||^2 of the current evaluation
    long long *sNext = reinterpret_cast<long long *>(smem_raw + (size_t)(kJS + Spec::NFACT + Spec::TSZ + 1) * SLOTS * sizeof(T)) + slot;

    // One-trip-ahead refill (arrow specs).  The SOLVER role learns in the middle of a trip -- behind the barrier inside
    // psolve() -- that a slot's problem has converged, and pulls the slot's next ticket right there.  For a converged
    // problem the slot's target strip and the Jacobian rows of the other roles are dead from that point on (no step is
    // taken), so the same thread starts the copy of the NEXT problem into them at once (cp.async: the new targets into
    // sT, the new configuration into Spec::QSTAGE .. + NQ of the Jacobian strip) and waits for it before the group's next
    // barrier -- on the role that idles most of the trip.  At the end of the trip every role picks its coordinates out
    // of the staged configuration with shared-memory loads; the global round trip that used to end every trip of every
    // role (3-4 of a group's 32 slots refill per trip) is gone from the critical roles' path.  Slots that finish
    // without converging, carried stragglers and the TAIL launch take the direct path (load_problem).
    // TMEMJ bodies (the Jacobian rows in tensor memory) stage the configuration in the factor strip instead, one copy per
    // role in the role's OWN published contributions (Spec::qstage_l): they are dead from the second barrier on, and the
    // next store into them is the role's own phase 1, after its loads in program order -- the roles run unordered from the
    // top barrier to the one inside psolve(), so a slot another role stores first would race with the loads.  The copies
    // are issued behind the second barrier and waited for at the end of the trip (kStager below); every role picks its
    // coordinates up behind the barrier at the top of the next trip.
    constexpr bool kPrefetch = Spec::ARROW && NW > 1 && !Spec::CAPSOLO && (kTmemJ ? spec_qstage_l<Spec>::value : Spec::QSTAGE >= 0) && IKB_PREFETCH;
    auto stage_at = [&](int r) -> T * {                     // the staged configuration role r reads
        if constexpr (kTmemJ && kPrefetch) return sm + (kJS + Spec::qstage_l(r)) * SLOTS;
        else return sm + (kPrefetch ? Spec::QSTAGE : 0) * SLOTS;
    };
    constexpr long long kStagedBit = 1LL << 62;             // in *sNext: the ticket's problem is already staged
    bool staged = false;    // (TMEMJ) this slot's next problem waits in the staging slots for the top of the next trip
    // TMEMJ: the SOLVER role carries the longer trip (stop test, free-flyer step, mailbox), so the copies are issued by
    // another role -- right after the second barrier, when the ticket is visible and the contributions are dead -- which
    // waits for them at the end of its trip, in the slack it used to spend at the barrier at the top of the loop
    constexpr int kStager = kTmemJ ? (Spec::SOLVER + 1) % NW : Spec::SOLVER;
    auto stage = [&](long long idx) {
        const ProblemIO<T> io = problem_io<SEG>(a, idx);
#pragma unroll
        for (int r = 0; r < NW; ++r) Spec::load_targets(r, io.targets, io.tg_es, sT);
#pragma unroll
        for (int r = 0; r < (kTmemJ ? NW : 1); ++r) {
            const S sQ{stage_at(r)};
#pragma unroll
            for (int k = 0; k < NQ; ++k) sQ.copy_in(k, io.q0 + k * io.q0_es);
        }
    };

    auto group_sync = [&]() {
        if constexpr (NW > 1)
            asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(NW * 32) : "memory");
        else
            __syncwarp();
    };

    T q[Spec::NQL];                                       // (arrow specs: only the coordinates this role reads and steps)
    // FP64 arrow kernels: q lives in tensor memory (32 columns of this thread's lane) whenever no phase needs it -- in
    // registers only from the top of a trip to the end of evaluate, and from the step to the end of the trip
    constexpr bool kTmemQ = IKB_TMEM_Q && Spec::ARROW && sizeof(T) == 8 && Spec::NQL <= 16;
    constexpr int kTmemCols = spec_tmem_cols<Spec, T>(GROUPS * NW);
    uint32_t tmem_base = 0, tmem_q = 0;
    if constexpr (kTmemQ) {
        static_assert(spec_tmem_quarter<Spec, T>(0, GROUPS * NW) <= 512 && spec_tmem_quarter<Spec, T>(1, GROUPS * NW) <= 512 &&
                      spec_tmem_quarter<Spec, T>(2, GROUPS * NW) <= 512 && spec_tmem_quarter<Spec, T>(3, GROUPS * NW) <= 512,
                      "the warps of one lane quarter need more than 512 tensor-memory columns");
        tmem_base = tmem_provision<kTmemCols>(reinterpret_cast<uint32_t *>(smem_raw), warp);
        uint32_t col = 0;                                   // the columns of the warps before this one in its lane quarter
        for (int w = warp & 3; w < warp; w += 4) col += (uint32_t)spec_tmem_width<Spec, T>(w % NW);
        tmem_q = tmem_base + ((uint32_t)(warp & 3) * 32u << 16) + col;   // lane quarter | first column of this warp
    }
    // weighted task Jacobian, non-zeros only: a shared-memory strip, or the role's own slots in tensor memory
    using SJ = typename std::conditional<kTmemJ, TStrip<double>, S>::type;
    SJ sJ;
    if constexpr (kTmemJ) sJ.base = tmem_q + 32u - 2u * (uint32_t)Spec::j_first(role);
    else sJ.base = sm;
    long long b;
    int it = 0;
    bool have;
    bool refetch = false;   // Spec::QCOMMON: this slot's problem was stepped in the last trip and goes on

    // b holds a ticket on entry: a problem index (fresh problems) or an index into the suspended list (tail launch)
    // (merged launches only) the stragglers carried over from the previous launch take the first tickets
    long long ncarry = 0;
    if constexpr (SEG)
        if (a.carry_list) ncarry = (long long)*a.carry_count;
    bool carried = false;   // this slot's problem is one of them: it lives in the previous launch's buffers
    auto pio = [&](long long idx) -> ProblemIO<T> {
        if constexpr (SEG)
            if (carried) return segment_io<T>(a.cseg, idx);
        return problem_io<SEG>(a, idx);
    };
    auto load_problem = [&]() {
        it = 0;
        refetch = false;
        carried = false;
        if (!a.resume) {
            if (SEG && b < ncarry) {
                carried = true;
                have = true;
                b = a.carry_list[b];
                it = a.carry_iters[b];
            } else {
                b -= ncarry;
                have = b < a.B;
            }
        } else {
            have = b < (long long)*a.list_count;
            if (have) {
                b = a.list[b];
                it = a.iters_ws[b];
            }
        }
        if (have) {
            const ProblemIO<T> io = pio(b);
            const T *src = (a.resume || carried) ? io.q : io.q0;       // a suspended problem continues from its saved iterate
            const long long es = (a.resume || carried) ? io.q_es : io.q0_es;
            Spec::load_targets(role, io.targets, io.tg_es, sT);   // cp.async: the whole pose in flight at once ...
            Spec::load_q(role, src, es, q);                        // ... under the loads of the configuration
            strip_copies_wait();
        }
    };
    // SOLVER role, after the solve: dq = -J^T y, the manifold step and the clamp on ITS copy of q, which it then publishes
    // in the (dead) factor strip -- the other roles only copy it (no second and third integrate on the critical path).
    auto step_and_publish = [&](const T(&y)[M], T sres) {
        if constexpr (!Spec::DSTEP)
        if (!(abs_(sres) < a.tolerance)) {                           // dls.cpp:61-64: a converged iterate is returned as is
            T dq[NV];
            Spec::step_direction(sJ, y, dq);                         // dls.cpp:52
            Spec::integrate(q, dq, a.step_length, c);                // dls.cpp:67-71
            if constexpr (NW > 1) {
#pragma unroll
                for (int k = 0; k < NQ; ++k) sD.set(k, q[k]);
            }
        }
        *sRes = sres;
    };

    // first ticket of every slot (the SOLVER role owns the ticket counter)
    if (role == Spec::SOLVER) *sNext = (long long)atomicAdd(a.ticket, 1ULL);
    group_sync();
    b = *sNext;
    load_problem();
    if constexpr (kTmemQ) tmem_park(tmem_q, q);

    // CTA-wide barrier at the top of every trip: the body is ~100 KB of straight-line code, far more than the 32 KB
    // instruction cache in front of L2, so every warp streams it from L2 on every trip.  Warps that start a trip together
    // stay in step (same instruction count whatever their lanes do) and share each fetched line; left alone they drift
    // apart and each pulls its own copy (ncu: no_instruction stalls 0.4 -> 1.1 per issue).
    auto any_left = [&]() -> bool {
        if (GROUPS == 1 || a.loop_sync == 1) return __syncthreads_or(have) != 0;
        if constexpr (NW > 1) {   // the group's own barrier with an OR reduction (bar.red on a named barrier)
            unsigned r;
            asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 q, %1, 0;\n\tbar.red.or.pred p, %2, %3, q;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(r) : "r"((unsigned)have), "r"(group + 1), "n"(NW * 32) : "memory");
            return r != 0;
        } else {
            return __any_sync(0xffffffffu, have) != 0;
        }
    };
    constexpr bool kTripProf = IKB_TRIP_PROFILE && kTmemJ && SEG;
    TripClock tc;
    auto tmark = [&](int seg) {
        if constexpr (kTripProf) tc.mark(seg);
    };
    if constexpr (kTripProf) tc.start();
    while (any_left()) {
        tmark(kTripTopBarrier);
        if constexpr (kTripProf) tc.trip();
        if constexpr (kTmemQ) tmem_fetch(tmem_q, q);        // (all lanes: the transfer is warp-wide)
        if constexpr (kPrefetch && kTmemJ) {
            if (__any_sync(0xffffffffu, staged)) {          // landed: the staging role waited before the barrier
                if (staged) Spec::load_q(role, stage_at(role), (long long)SLOTS, q);
                tmem_park(tmem_q, q);                       // (warp-wide) the step fetches q from tensor memory again
            }
            staged = false;
        }
        tmark(kTripTmemFetch);
        if constexpr (Spec::QCOMMON) {
            if (have && refetch) Spec::fetch_common(role, sL, q);   // the coordinates the solver role stepped for everybody
            refetch = false;
        }
        if constexpr (kTmemJ) {
            // tensor-memory transfers are warp-wide (.sync.aligned): every lane evaluates, also the ones without a problem
            // (on stale or arbitrary inputs; nobody reads what they produce)
            Spec::evaluate(role, q, sT, c, sJ, sE);
            sJ.flush();
            tmark(kTripEvaluate);
        } else if (have) {
            Spec::evaluate(role, q, sT, c, sJ, sE);         // data.cpp:25-58, this role's tasks
            // The solver role's own tasks are the cheap ones: while the others still evaluate, it factorises the leading
            // block of the normal equations, which involves its rows only (off the critical path, no extra barrier).
            if constexpr (Spec::PRE > 0)
                if (role == Spec::SOLVER) Spec::presolve(sJ, sL, sE, a.damping2);
        }
        // (an ARROW step starts with role-local work on the role's own rows: it needs no barrier here, and its stop test
        // runs as a hook behind the one barrier inside psolve())
        if constexpr (!Spec::ARROW) group_sync();           // J and e of all roles visible
        T sres_mine = T(0);
        auto stop_test = [&]() {
            if (role == Spec::SOLVER && have) {
            // The stop-test quantity first: a slot that is about to finish (converged, or on its last iteration) pulls
            // its next ticket NOW, so the atomic's latency hides behind the solve and no slot ever hoards a ticket.
            T res = T(0);
#pragma unroll
            for (int i = 0; i < Spec::M0; ++i) {
                const T ei = sE.get(i);
                res += ei * ei;                                     // visitor.hpp:19 (priority-0 rows)
            }
            // Bulk launch only: once the ticket queue has run dry, a problem that has already taken it_cap steps is a
            // straggler -- suspend it after this step and let the tail launch continue it (res >= tolerance > 0 here, so
            // the decision travels to the other roles in the sign of the residual).
            bool susp = false;
            if (it + 1 >= a.it_cap && !(res < a.tolerance) && it + 1 < a.max_iterations && !carried)
                susp = *(volatile unsigned long long *)a.ticket >= (unsigned long long)(a.B + ncarry);
            if (res < a.tolerance || it + 1 >= a.max_iterations || susp) {
                long long nb = (long long)atomicAdd(a.ticket, 1ULL);
                if constexpr (kPrefetch) {
                    if (res < a.tolerance && !a.resume && nb >= ncarry && nb - ncarry < a.B) {   // converged here, a fresh problem next
                        if constexpr (!kTmemJ) stage(nb - ncarry);
                        nb |= kStagedBit;
                    }
                }
                *sNext = nb;
            }
            sres_mine = susp ? -res : res;
            if constexpr (Spec::ARROW) *sRes = sres_mine;
            }
        };
        if constexpr (!Spec::ARROW) stop_test();
        if constexpr (NW > 1 && Spec::ARROW) {
            // Bordered-block-diagonal step (gen_solve_arrow): phase 1 on the role's own rows, ONE barrier, the stop test
            // (solver role, all of e visible), the small shared-column system in every role, y for the role's own rows.
            T y[Spec::MY];
            if constexpr (kTripProf) {
                auto sync1 = [&]() {
                    group_sync();
                    tmark(kTripPhase1);
                };
                auto hook = [&]() {
                    stop_test();
                    tmark(kTripStopTest);
                };
                Spec::psolve(role, sJ, sL, sE, a.damping2, y, sync1, hook);
                tmark(kTripPhase23);
            } else {
                Spec::psolve(role, sJ, sL, sE, a.damping2, y, group_sync, stop_test);
            }
            if constexpr (kPrefetch && !kTmemJ)
                if (role == Spec::SOLVER) strip_copies_wait();   // the staged problems have landed before the others look
            if constexpr (!Spec::CAPSOLO) group_sync();     // s and ||e||^2 visible (y is role-private)
            tmark(kTripBarrier2);
            if constexpr (kPrefetch && kTmemJ)
                if (role == kStager && have && abs_(*sRes) < a.tolerance) {   // converged: *sNext is this trip's ticket
                    const long long nb = *sNext;
                    if (nb & kStagedBit) stage((nb & ~kStagedBit) - ncarry);
                }
            if constexpr (kTmemQ) tmem_fetch(tmem_q, q);    // back for the step (a non-solver role's copy of the common
                                                            // coordinates is stale here: it neither steps nor stores them)
            if constexpr (kTmemJ) {
                // (warp-wide again: every lane steps a copy, the lanes whose problem goes on keep it)
                T qn[Spec::NQL];
#pragma unroll
                for (int k = 0; k < Spec::NQL; ++k) qn[k] = q[k];
                if constexpr (Spec::MY != M) Spec::step_role(role, sJ, sL, qn, a.step_length, c, y);
                else Spec::step_role(role, sJ, sL, qn, a.step_length, c);
                const bool go = have && !(abs_(*sRes) < a.tolerance);
#pragma unroll
                for (int k = 0; k < Spec::NQL; ++k) q[k] = go ? qn[k] : q[k];
                if (go) refetch = true;
                tmark(kTripStep);
            } else if (have && !(abs_(*sRes) < a.tolerance)) {     // dls.cpp:52,61-71
                if constexpr (Spec::MY != M) Spec::step_role(role, sJ, sL, q, a.step_length, c, y);   // y in the role's registers
                else Spec::step_role(role, sJ, sL, q, a.step_length, c);
                refetch = true;
            }
        } else if constexpr (NW > 1 && Spec::PSOLVE) {
            // dls.cpp:39-41,53 distributed over the roles (cyclic row ownership, two barriers per block column).  Every
            // lane of every warp takes part in the barriers, also lanes without a problem (their arithmetic is garbage
            // that nobody reads).
            T y[M];
            Spec::psolve(role, sJ, sL, sE, a.damping2, y, group_sync);
            if constexpr (Spec::DSTEP) {
                // Distributed step: y is in the strip; every role takes dq = -J^T y and the manifold step on the
                // coordinates its own evaluate reads (the free-flyer redundantly, with the same instructions), so the
                // solver role's serial tail -- 40 % of a humanoid iteration in the ncu profile -- shrinks to the back
                // substitution.  One more barrier: y and ||e||^2 visible.
                if (role == Spec::SOLVER && have) *sRes = sres_mine;
                group_sync();
                if (have && !(abs_(*sRes) < a.tolerance)) Spec::step_role(role, sJ, sL, q, a.step_length, c);  // dls.cpp:52,61-71
            } else {
                if (role == Spec::SOLVER && have) step_and_publish(y, sres_mine);
            }
        } else {
            if (role == Spec::SOLVER && have) {
                T y[M];
                Spec::solve(sJ, sL, sE, a.damping2, y);             // dls.cpp:39-41,53
                step_and_publish(y, sres_mine);
            }
        }
        // (ARROW: nothing a role writes from here to the CTA-wide barrier at the top of the loop is read by another role)
        if constexpr (!Spec::ARROW) group_sync();           // ||e||^2, dq (and the next ticket) visible; J, e, factor dead
        [[maybe_unused]] long long tp_refill = 0;   // (IKB_TRIP_PROFILE)
        if (have) {
            const T sres = *sRes;
            const bool suspend = sres < T(0);               // bulk launch: hand the straggler to the tail launch
            const T res = abs_(sres);
            const bool converged = res < a.tolerance;       // visitor.hpp:19
            bool finished = converged;                      // dls.cpp:61-64: the un-stepped iterate is returned
            if (!converged) {
                if constexpr (NW > 1 && !Spec::DSTEP) {
                    if (role != Spec::SOLVER) {             // the stepped, clamped iterate (dls.cpp:67-71) from the solver
#pragma unroll
                        for (int k = 0; k < NQ; ++k) q[k] = sD.get(k);
                    }
                }
                ++it;
                finished = it >= a.max_iterations;          // dls.cpp:14,76-77
            }
            if (finished || suspend) {
                if constexpr (Spec::DSTEP) {                // every role holds (and writes) its own coordinates
                    const ProblemIO<T> io = pio(b);
                    Spec::store_q(role, q, io.q, io.q_es);
                }
                if (role == Spec::SOLVER) {
                    const ProblemIO<T> io = pio(b);
                    if constexpr (!Spec::DSTEP) {
#pragma unroll
                        for (int k = 0; k < NQ; ++k) io.q[k * io.q_es] = q[k];
                    }
                    if (suspend) {
                        a.iters_ws[b] = it;
                        a.list[atomicAdd(a.list_count, 1ULL)] = (unsigned int)b;
                    } else {
                        if (io.success) *io.success = converged ? 1 : 0;
                        if (io.iters) *io.iters = it;
                        if (io.resid) *io.resid = res;
                    }
                }
                if constexpr (kTripProf) tp_refill = clock64();
                b = *sNext;
                if constexpr (kPrefetch) {
                    if (b & kStagedBit) {                    // staged during this trip
                        b = (b & ~kStagedBit) - ncarry;
                        it = 0;
                        refetch = false;
                        carried = false;
                        have = true;
                        if constexpr (kTmemJ) staged = true;     // (the copies may still be in flight)
                        else Spec::load_q(role, stage_at(0), (long long)SLOTS, q);
                    } else {
                        load_problem();
                    }
                } else {
                    load_problem();
                }
            }
        }
        if constexpr (kPrefetch && kTmemJ)
            if (role == kStager) strip_copies_wait();       // the staged problems land before the barrier at the top
        if constexpr (kTripProf) tc.split(tp_refill);
        if constexpr (kTmemQ) tmem_park(tmem_q, q);         // stepped, refilled or unchanged: out of the registers again
        tmark(kTripPark);
    }
    if constexpr (kTripProf) {
        tmark(kTripTopBarrier);
        tc.flush(role);
    }
    if constexpr (kTmemQ) tmem_release<kTmemCols>(tmem_base, warp);
}

// ---- host side ------------------------------------------------------------------------------------------

inline bool same_values(const double *a, const double *b, int n) {  // value equality (-0.0 == 0.0), not bit equality
    for (int i = 0; i < n; ++i)
        if (!(a[i] == b[i])) return false;
    return true;
}

// Specs with a centre-of-mass task fold every joint's mass and centre of mass into their code and carry them as
// Spec::sig_inertia() (mass, com x, y, z per joint); the other generated headers have no such member.
template <class Spec, class = void> struct spec_has_inertia : std::false_type {};
template <class Spec> struct spec_has_inertia<Spec, std::void_t<decltype(Spec::sig_inertia())>> : std::true_type {};

// Specs generated with FrameConstraints project every step onto their null space and carry the constraint list as
// Spec::sig_con_type() etc. (NCONS entries in stacked order); the other generated headers have no such member.
template <class Spec, class = void> struct spec_has_constraints : std::false_type {};
template <class Spec> struct spec_has_constraints<Spec, std::void_t<decltype(Spec::sig_con_type())>> : std::true_type {};

// Does the problem's constraint list have the Spec's structure: count, order, type, frame and reference joints?
// (A Spec without constraints: only an empty list.)
template <class Spec> bool spec_constraint_structure(const HostProblem &hp) {
    if constexpr (spec_has_constraints<Spec>::value) {
        if ((int)hp.constraints.size() != Spec::NCONS) return false;
        const HostModel &m = hp.model;
        for (int k = 0; k < Spec::NCONS; ++k) {
            const HostConstraint &hc = hp.constraints[k];
            if (hc.type != Spec::sig_con_type()[k] || m.frame_parent[hc.frame] != Spec::sig_con_joint()[k] ||
                m.frame_parent[hc.ref] != Spec::sig_con_ref_joint()[k])
                return false;
        }
        return true;
    } else {
        return hp.constraints.empty();
    }
}

// generator task kind code (sig_task_kind) -> HostTask::kind
constexpr int kSpecTaskKinds[4] = {IKB_TASK_FRAME, IKB_TASK_ALIGN_AXIS, IKB_TASK_POSTURE, IKB_TASK_COM};

// Does the finalized problem equal the (tree, task list) this specialisation was generated for?
template <class Spec> bool spec_matches(const HostProblem &hp) {
    const HostModel &m = hp.model;
    if (m.njoints() != Spec::NJOINTS || m.nq != Spec::NQ || m.nv != Spec::NV) return false;
    if ((int)hp.tasks.size() != Spec::NTASKS || hp.rows() != Spec::M || hp.e_size(0) != Spec::M0) return false;
    const int *par = Spec::sig_parent(), *typ = Spec::sig_type();
    const double *pl = Spec::sig_placement();
    for (int j = 0; j < Spec::NJOINTS; ++j) {
        if (m.parent[j] != par[j] || m.jtype[j] != typ[j]) return false;
        if (!same_values(m.placement[j].data(), pl + 15 * j, 12)) return false;
        if (typ[j] > IKB_J_FREEFLYER && axis_index(typ[j]) < 0)   // unaligned: the axis is part of the model
            if (!same_values(m.axis[j].data(), pl + 15 * j + 12, 3)) return false;
    }
    // the inertias the com task's code was generated with (ikb_model_set_inertias).  Every joint is compared, the massless
    // `universe` (joint 0) too, although no centre of mass reads its entry: tools/com_plugin_bench.py tells two plugins of
    // one task list apart by it.
    if constexpr (spec_has_inertia<Spec>::value) {
        const double *in = Spec::sig_inertia();
        for (int j = 0; j < Spec::NJOINTS; ++j)
            if (!(m.mass[j] == in[4 * j]) || !same_values(m.com[j].data(), in + 4 * j + 1, 3)) return false;
    }
    // tasks must already be in stacked order (the generated code has no notion of insertion order)
    for (int t = 0; t < Spec::NTASKS; ++t) {
        const HostTask &ht = hp.tasks[t];
        if (ht.kind != kSpecTaskKinds[Spec::sig_task_kind()[t]]) return false;
        if (ht.type != Spec::sig_task_type()[t] || ht.priority != Spec::sig_task_priority()[t]) return false;  // type / axis / nj
        if (t > 0 && ht.priority < hp.tasks[t - 1].priority) return false;
        if (ht.kind == IKB_TASK_POSTURE) continue;  // no frames
        // the reference frame (`universe` or a moving frame) and the task frame must sit where the generator saw them
        // (a centre-of-mass task has no frame of its own: HostTask::frame is its reference frame)
        if (m.frame_parent[ht.ref] != Spec::sig_task_ref_joint()[t]) return false;
        if (!same_values(m.frame_placement[ht.ref].data(), Spec::sig_task_ref_placement() + 12 * t, 12)) return false;
        if (m.frame_parent[ht.frame] != Spec::sig_task_joint()[t]) return false;
        if (!same_values(m.frame_placement[ht.frame].data(), Spec::sig_task_placement() + 12 * t, 12)) return false;
    }
    // the constraints, in the order Jc stacks them, with the frame placements their code was generated for
    if (!spec_constraint_structure<Spec>(hp)) return false;
    if constexpr (spec_has_constraints<Spec>::value) {
        for (int k = 0; k < Spec::NCONS; ++k) {
            const HostConstraint &hc = hp.constraints[k];
            if (!same_values(m.frame_placement[hc.frame].data(), Spec::sig_con_placement() + 12 * k, 12)) return false;
            if (!same_values(m.frame_placement[hc.ref].data(), Spec::sig_con_ref_placement() + 12 * k, 12)) return false;
        }
    }
    return true;
}

// Near miss: the problem has this specialisation's topology, joint types and task list, but some placement differs
// (slightly: a re-rounded URDF literal; or grossly: another robot of the same shape) from the values the straight-line
// code was generated with, so spec_matches rejected it.  `why` names the first difference and its size.
template <class Spec> bool spec_near_miss(const HostProblem &hp, std::string *why) {
    const HostModel &m = hp.model;
    if (m.njoints() != Spec::NJOINTS || m.nq != Spec::NQ || m.nv != Spec::NV) return false;
    if ((int)hp.tasks.size() != Spec::NTASKS || hp.rows() != Spec::M || hp.e_size(0) != Spec::M0) return false;
    if (!spec_constraint_structure<Spec>(hp)) return false;
    const int *par = Spec::sig_parent(), *typ = Spec::sig_type();
    for (int j = 0; j < Spec::NJOINTS; ++j)
        if (m.parent[j] != par[j] || m.jtype[j] != typ[j]) return false;
    for (int t = 0; t < Spec::NTASKS; ++t) {
        const HostTask &ht = hp.tasks[t];
        if (ht.kind != kSpecTaskKinds[Spec::sig_task_kind()[t]] || ht.type != Spec::sig_task_type()[t] || ht.priority != Spec::sig_task_priority()[t]) return false;
        if (ht.kind == IKB_TASK_POSTURE) continue;
        if (m.frame_parent[ht.ref] != Spec::sig_task_ref_joint()[t] || m.frame_parent[ht.frame] != Spec::sig_task_joint()[t]) return false;
    }
    // same structure: find the largest numeric difference
    double worst = 0;
    char where[160] = "";
    auto scan = [&](const double *a, const double *b, int n, const char *what, int idx, const char *name) {
        for (int i = 0; i < n; ++i) {
            const double d = a[i] > b[i] ? a[i] - b[i] : b[i] - a[i];
            if (d > worst) {
                worst = d;
                std::snprintf(where, sizeof where, "%s %d (%s), entry %d: %.17g here vs %.17g generated", what, idx, name, i, a[i], b[i]);
            }
        }
    };
    const double *pl = Spec::sig_placement();
    for (int j = 0; j < Spec::NJOINTS; ++j) {
        scan(m.placement[j].data(), pl + 15 * j, 12, "placement of joint", j, m.joint_names[j].c_str());
        if (typ[j] > IKB_J_FREEFLYER && axis_index(typ[j]) < 0) scan(m.axis[j].data(), pl + 15 * j + 12, 3, "axis of joint", j, m.joint_names[j].c_str());
    }
    for (int t = 0; t < Spec::NTASKS; ++t) {
        const HostTask &ht = hp.tasks[t];
        if (ht.kind == IKB_TASK_POSTURE) continue;
        scan(m.frame_placement[ht.ref].data(), Spec::sig_task_ref_placement() + 12 * t, 12, "reference frame of task", t, m.frame_names[ht.ref].c_str());
        scan(m.frame_placement[ht.frame].data(), Spec::sig_task_placement() + 12 * t, 12, "frame of task", t, m.frame_names[ht.frame].c_str());
    }
    if constexpr (spec_has_constraints<Spec>::value) {
        for (int k = 0; k < Spec::NCONS; ++k) {
            const HostConstraint &hc = hp.constraints[k];
            scan(m.frame_placement[hc.frame].data(), Spec::sig_con_placement() + 12 * k, 12, "frame of constraint", k, m.frame_names[hc.frame].c_str());
            scan(m.frame_placement[hc.ref].data(), Spec::sig_con_ref_placement() + 12 * k, 12, "reference frame of constraint", k, m.frame_names[hc.ref].c_str());
        }
    }
    if (!(worst > 0)) return false;   // equal values: not a miss at all (IKB_FORCE_GENERIC, task order, ...)
    if (why) {
        char buf[400];
        std::snprintf(buf, sizeof buf, "specialisation '%s' has this problem's topology and task list but was generated for other placements "
                      "(largest difference %.3g: %s); running the table-driven kernel", Spec::name(), worst, where);
        *why = buf;
    }
    return true;
}

// GROUPS = 32-problem groups per CTA, MINB = CTAs per SM the register allocation must allow.  The throughput
// configuration is one big CTA per SM (GROUPS = SpecLaunch::GROUPS); the latency configuration is GROUPS = 1, so that
// few problems spread over all SMs and every group has its schedulers to itself.
template <class Spec, typename T, int GROUPS, int MINB, bool SEG>
int launch_spec_cfg_seg(const SpecHostConsts &hc, const SolveArgs<T> &a, long long ctas, cudaStream_t s) {
    using L = SpecLaunch<Spec, T>;
    static_assert(L::kFits && GROUPS <= L::GROUPS, "per-problem strips do not fit in shared memory for this scalar type");
    constexpr int kSmem = L::smem_bytes(GROUPS);
    auto fn = dls_spec_kernel<Spec, T, GROUPS, MINB, SEG>;
    static DynSmemOptIn opt_in;  // per instantiation; the attribute itself is per DEVICE
    if (!opt_in.ensure(fn, kSmem)) return 1;
    SpecConsts<T, Spec::NQ, Spec::M> c;
    for (int k = 0; k < Spec::NQ; ++k) {
        c.lower[k] = (T)hc.lower[k];
        c.upper[k] = (T)hc.upper[k];
    }
    for (int i = 0; i < Spec::M; ++i) {
        c.weight[i] = (T)hc.weight[i];
        c.mask[i] = (T)hc.mask[i];
    }
    if (ctas < 1) ctas = 1;
    SolveArgs<T> a2 = a;
    if (const char *e = std::getenv("IKB_LOOP_SYNC")) a2.loop_sync = e[0] == 'c' ? 1 : 0;   // cta | group (A/B runs)
    fn<<<(unsigned)ctas, GROUPS * Spec::NWARPS * 32, kSmem, s>>>(c, a2);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

template <class Spec, typename T, int GROUPS, int MINB>
int launch_spec_cfg(const SpecHostConsts &hc, const SolveArgs<T> &a, long long ctas, cudaStream_t s) {
    return a.nseg > 0 ? launch_spec_cfg_seg<Spec, T, GROUPS, MINB, true>(hc, a, ctas, s)
                 : launch_spec_cfg_seg<Spec, T, GROUPS, MINB, false>(hc, a, ctas, s);
}

// Throughput configuration: persistent, one CTA per SM.
template <class Spec, typename T> int launch_spec_bulk(const SpecHostConsts &hc, const SolveArgs<T> &a, long long n, int sm_count, cudaStream_t s) {
    using L = SpecLaunch<Spec, T>;
    long long ctas = (n + L::GROUPS * 32 - 1) / (L::GROUPS * 32);
    if (ctas > sm_count) ctas = sm_count;
    return launch_spec_cfg<Spec, T, L::GROUPS, 1>(hc, a, ctas, s);
}
// Latency configuration: one 32-problem group per CTA, at most 2 CTAs per SM (full register budget per thread).
template <class Spec, typename T> int launch_spec_tail(const SpecHostConsts &hc, const SolveArgs<T> &a, long long n, int sm_count, cudaStream_t s) {
    using L = SpecLaunch<Spec, T>;
    // two CTAs per SM only if shared memory allows it and every thread still gets the full 255-register budget
    constexpr int kPerSm = (2 * (L::smem_bytes(1) + 1024) <= 228 * 1024 && 2 * Spec::NWARPS * 32 * 255 <= 65536) ? 2 : 1;
    long long ctas = (n + 31) / 32;
    if constexpr (kPerSm == 2) {
        // more groups than SMs: IKB_TAIL_PAIR=1 pairs them in one CTA that starts every trip together, so that the two groups
        // share the instruction lines they fetch (a lone group streams ~40 KB of straight-line code per trip).  Off by
        // default: 40 interleaved lone batches (tools/pair_ab.py, profiles/r2_s4_pair_ab.txt) take 0.811 ms with two
        // independent one-group CTAs per SM against 0.840 ms paired -- the lock step costs more than the shared fetch saves.
        const char *e = std::getenv("IKB_TAIL_PAIR");
        if (ctas > sm_count && e && e[0] == '1') {
            ctas = (ctas + 1) / 2;
            if (ctas > sm_count) ctas = sm_count;
            SolveArgs<T> a2 = a;
            a2.loop_sync = 1;
            return launch_spec_cfg<Spec, T, 2, 1>(hc, a2, ctas, s);
        }
    }
    if (ctas > (long long)kPerSm * sm_count) ctas = (long long)kPerSm * sm_count;
    return launch_spec_cfg<Spec, T, 1, kPerSm>(hc, a, ctas, s);
}

}  // namespace ikb
