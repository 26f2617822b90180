// Specialised solve kernels: Cassie (free-flyer) with pelvis Full + LeftFootFront / RightFootFront Position tasks in
// `universe` -- the BASELINE.json headline problem (reference task set-up: ik_ros/src/cassie.cpp:43-81).
//
// BULK (throughput): thread-per-problem, generated arithmetic; three decompositions are compiled
// (ik_b200/specs/cassie_feet_pelvis*.json): one warp role (W1), two (pelvis+left | right+solve, W2) and three
// (pelvis+solve | left | right, W3, with presolve); W3 is the measured-best one for both scalar types, IKB_CASSIE_ROLES=1|2|3
// overrides it (tools/bench_variants.sh).  The merged FP64 BULK launch of W3 runs the arrow step with the pelvis folded into
// the two leg roles (cassie_feet_pelvis_fold: 6 groups = 192 problems per SM, Jacobian rows in tensor memory).
// TAIL (latency): the team-per-problem kernel of dls_team.cuh -- 16 lanes share one problem -- for the stragglers a BULK
// launch suspends and for batches too small to fill the GPU.  IKB_CASSIE_TAIL=0 selects the previous latency
// configuration (W3, one 32-problem group per CTA) for A/B measurements.
#include <cstdlib>
#include <cstring>

#include "dls_spec.cuh"
#include "dls_team.cuh"
#include "gen/cassie_feet_pelvis.cuh"
#include "gen/cassie_feet_pelvis_arrow.cuh"
#include "gen/cassie_feet_pelvis_arrow_b.cuh"
#include "gen/cassie_feet_pelvis_fold.cuh"
#include "gen/cassie_feet_pelvis_w1.cuh"
#include "gen/cassie_feet_pelvis_w2.cuh"

namespace ikb {
namespace {
using S3 = SpecCassieFeetPelvis;
using SA = SpecCassieFeetPelvisArrow;  // three roles, bordered-block-diagonal step (gen_solve_arrow) instead of the dense 12 x 12 solve
using S2 = SpecCassieFeetPelvisW2;
using S1 = SpecCassieFeetPelvisW1;
using SB = SpecCassieFeetPelvisArrowB;  // ... factor / y in registers, free-flyer stepped once by the pelvis role
// ... two roles (left | right leg), each evaluating the pelvis pose in registers and publishing half of its share of the
// shared-column system: no idle pelvis warp, so 6 groups of 2 warps fit where 4 groups of 3 did (same arithmetic as SA)
using SF = SpecCassieFeetPelvisFold;
// IKB_CASSIE_SOLVE=dense|arrow|arrowb|fold (A/B runs).  (Solving the shared-column system on the pelvis role alone --
// spec option arrow_cap_solo -- was measured too: 3.13 ms against 3.10 ms for 8 x 65 536, not kept.)
int solve_variant(bool f64, bool tail) {
    const char *e = std::getenv("IKB_CASSIE_SOLVE");
    if (e && std::strcmp(e, "dense") == 0) return 0;
    if (e && std::strcmp(e, "arrow") == 0) return 1;
    if (e && std::strcmp(e, "arrowb") == 0) return 2;
    if (e && std::strcmp(e, "fold") == 0) return 3;
    // the throughput launch in FP64 is register-bound (168 per thread): factor in shared memory, pelvis folded into the
    // leg roles; everything else has registers to spare (the arrow variants run the same arithmetic: bit-identical results)
    return (f64 && !tail) ? 3 : 2;
}
int roles(int dflt) {
    const char *e = std::getenv("IKB_CASSIE_ROLES");
    return (e && e[0] >= '1' && e[0] <= '3') ? e[0] - '0' : dflt;
}

// The team kernel's view of the tree, read from the generated specialisation's signature: limb l = the chain of joints
// between the free-flyer and the frame of task 1 + l.  Its lane <-> joint map needs joint 2 + 8 l + (k < 6 ? k : 7) to be
// chain joint k of limb l, every chain joint a z-axis revolute and the base task frame to be the free-flyer frame.
struct TeamTree {
    bool ok = false;
    int chain[2][kTeamChain];
    TeamTree() {
        if (S3::NJOINTS != 18 || S3::NTASKS != 3 || S3::NQ != 23 || S3::M != 12) return;
        const int *par = S3::sig_parent(), *typ = S3::sig_type(), *tj = S3::sig_task_joint(), *tt = S3::sig_task_type();
        if (tj[0] != 1 || typ[1] != IKB_J_FREEFLYER || tt[0] != IKB_FULL || tt[1] != IKB_POSITION || tt[2] != IKB_POSITION) return;
        const double *fp = S3::sig_task_placement();
        for (int i = 0; i < 12; ++i)
            if (fp[i] != ((i == 0 || i == 4 || i == 8) ? 1.0 : 0.0)) return;
        for (int l = 0; l < 2; ++l) {
            int j = tj[1 + l], n = 0, rev[32];
            while (j > 1 && n < 32) {
                rev[n++] = j;
                j = par[j];
            }
            if (j != 1 || n != kTeamChain) return;
            for (int k = 0; k < kTeamChain; ++k) {
                chain[l][k] = rev[kTeamChain - 1 - k];
                if (typ[chain[l][k]] != IKB_J_RZ || chain[l][k] != 2 + 8 * l + (k < 6 ? k : 7)) return;
            }
        }
        ok = true;
    }
};
const TeamTree &team_tree() {
    static const TeamTree t;
    return t;
}
template <typename T> TeamConsts<T> team_consts(const SpecHostConsts &hc) {
    TeamConsts<T> c{};
    const TeamTree &t = team_tree();
    const double *pl = S3::sig_placement(), *fp = S3::sig_task_placement();
    for (int l = 0; l < 2; ++l) {
        for (int k = 0; k < kTeamChain; ++k) {
            const double *p = pl + 15 * t.chain[l][k];
            for (int i = 0; i < 9; ++i) c.PR[l][k][i] = (T)p[i];
            for (int i = 0; i < 3; ++i) c.Pp[l][k][i] = (T)p[9 + i];
        }
        for (int i = 0; i < 9; ++i) c.FR[l][i] = (T)fp[12 * (1 + l) + i];
        for (int i = 0; i < 3; ++i) c.Fp[l][i] = (T)fp[12 * (1 + l) + 9 + i];
    }
    for (int k = 0; k < S3::NQ; ++k) {
        c.lower[k] = (T)hc.lower[k];
        c.upper[k] = (T)hc.upper[k];
    }
    for (int i = 0; i < S3::M; ++i) c.weight[i] = (T)hc.weight[i];
    return c;
}
// Measured on B200 (profiles/r1_team_*.txt): the team kernel wins whenever latency binds -- every batch that fits the
// latency configuration (FP64 4 096: 0.73 -> 0.57 ms, FP32: 0.70 -> 0.41 ms) and the FP32 straggler launch (65 536: 0.92
// -> 0.66 ms).  The FP64 straggler launch of a large batch is the exception: ~4 500 problems x 16 lanes is FP64-pipe
// bound (a team spends ~4.5x the DFMA issue slots of a thread per problem-iteration), no faster than thread-per-problem.
bool use_team(bool is_f64, bool resume) {
    const char *e = std::getenv("IKB_CASSIE_TAIL");
    if (!team_tree().ok || (e && e[0] == '0')) return false;
    if (e && e[0] == 't') return true;
    return !(is_f64 && resume);
}

template <typename T> int launch(const SpecHostConsts &hc, const SolveArgs<T> &a, int variant, long long n, int sms, cudaStream_t s,
                                 int bulk_roles) {
    if (variant == SPEC_TAIL) {
        if (use_team(sizeof(T) == 8, a.resume != 0)) return launch_team<T>(team_consts<T>(hc), a, n, sms, s);
        switch (solve_variant(sizeof(T) == 8, true)) {
            case 0: return launch_spec_tail<S3, T>(hc, a, n, sms, s);
            case 1: return launch_spec_tail<SA, T>(hc, a, n, sms, s);
            case 3:
                if constexpr (sizeof(T) == 8) return launch_spec_tail<SF, T>(hc, a, n, sms, s);
                return launch_spec_tail<SB, T>(hc, a, n, sms, s);
            default: return launch_spec_tail<SB, T>(hc, a, n, sms, s);
        }
    }
    switch (roles(bulk_roles)) {
        case 3:
            switch (solve_variant(sizeof(T) == 8, false)) {
                case 0: return launch_spec_bulk<S3, T>(hc, a, n, sms, s);
                case 1: return launch_spec_bulk<SA, T>(hc, a, n, sms, s);
                case 3:   // (FP64 only: in FP32 the Jacobian rows would have to stay in shared memory)
                    // A merged launch of the queue (several batches) runs SF: 2.40 -> 2.09 ms per launch, 203 -> 230 M
                    // solves/s (B200).  A lone batch keeps SA: with SF its BULK + TAIL pair took 0.82 instead of 0.79 ms --
                    // 192 slots per SM still hold more problems when the queue runs dry, and the TAIL launch gets them.
                    if constexpr (sizeof(T) == 8) return a.nseg > 0 ? launch_spec_bulk<SF, T>(hc, a, n, sms, s) : launch_spec_bulk<SA, T>(hc, a, n, sms, s);
                    return launch_spec_bulk<SB, T>(hc, a, n, sms, s);
                default: return launch_spec_bulk<SB, T>(hc, a, n, sms, s);
            }
        case 2: return launch_spec_bulk<S2, T>(hc, a, n, sms, s);
        default: return launch_spec_bulk<S1, T>(hc, a, n, sms, s);
    }
}
int l64(const SpecHostConsts &hc, const SolveArgs<double> &a, int v, long long n, int sms, cudaStream_t s) {
    return launch<double>(hc, a, v, n, sms, s, 3);
}
int l32(const SpecHostConsts &hc, const SolveArgs<float> &a, int v, long long n, int sms, cudaStream_t s) {
    return launch<float>(hc, a, v, n, sms, s, 3);  // with presolve the 3-role split wins in FP32 too (156 vs 145 M solves/s merged)
}
}  // namespace
extern const SpecializedKernel kSpecCassieFeetPelvis = {S3::name(), spec_matches<S3>, l64, l32, spec_near_miss<S3>};
}  // namespace ikb

#if IKB_TRIP_PROFILE
// tools/trip_profile.py: copy out (and zero) the trip-segment counters of the merged fold launches (dls_spec.cuh, TripClock)
extern "C" int ikb_trip_profile(unsigned long long *out, int n) {
    static const unsigned long long zero[4 * (ikb::kTripSegs + 1)] = {};
    if (n * 8 > (int)sizeof(zero)) return 1;
    if (out && cudaMemcpyFromSymbol(out, ikb::ikb_trip_cycles, n * 8) != cudaSuccess) return 1;
    return cudaMemcpyToSymbol(ikb::ikb_trip_cycles, zero, sizeof(zero)) == cudaSuccess ? 0 : 1;
}
#endif
