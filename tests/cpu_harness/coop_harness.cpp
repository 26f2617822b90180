// TEST-ONLY: runs the table-driven team-per-problem iteration (ik_b200/csrc/dls_coop.cuh -- the very source the CUDA
// kernel dls_coop_kernel instantiates) on the CPU.  The TEAM lanes of a problem are ucontext fibers scheduled round
// robin: a lane that reaches a barrier yields, and is resumed once every other lane has yielded too, so __syncwarp and
// __shfl_sync keep their meaning.  The problem blob is filled by the product's own host code (urdf_model.cpp,
// problem_fill.hpp).  Never linked into libikb200.so; the product has no CPU path.
#include <ucontext.h>

#include <cstdio>
#include <cstring>
#include <functional>
#include <memory>
#include <string>
#include <vector>

#include "../../ik_b200/csrc/dls_coop.cuh"
#include "../../ik_b200/csrc/problem_fill.hpp"
#include "../../ik_b200/csrc/urdf_model.cpp"

using namespace ikb;

namespace {
struct FiberTeam {
    int n = 0, cur = 0;
    ucontext_t main_ctx;
    std::vector<ucontext_t> ctx;
    std::vector<std::unique_ptr<char[]>> stacks;
    std::vector<char> done;
    std::function<void(int)> body;
    static FiberTeam *self;
    static void trampoline() {
        FiberTeam *t = self;
        const int lane = t->cur;
        t->body(lane);
        t->done[lane] = 1;
        swapcontext(&t->ctx[lane], &t->main_ctx);
    }
    void run(int lanes, std::function<void(int)> f) {
        n = lanes;
        body = std::move(f);
        ctx.resize(n);
        done.assign(n, 0);
        stacks.clear();
        const size_t kStack = 1 << 20;
        for (int i = 0; i < n; ++i) {
            stacks.emplace_back(new char[kStack]);
            getcontext(&ctx[i]);
            ctx[i].uc_stack.ss_sp = stacks[i].get();
            ctx[i].uc_stack.ss_size = kStack;
            ctx[i].uc_link = &main_ctx;
            makecontext(&ctx[i], trampoline, 0);
        }
        self = this;
        for (;;) {
            bool any = false;
            for (int i = 0; i < n; ++i) {
                if (done[i]) continue;
                any = true;
                cur = i;
                swapcontext(&main_ctx, &ctx[i]);
            }
            if (!any) break;
        }
    }
    void yield() { swapcontext(&ctx[cur], &main_ctx); }
};
FiberTeam *FiberTeam::self = nullptr;

struct HostCtx {
    int lane;
    FiberTeam *team;
    double *xd;
    float *xf;
    void sync() const { team->yield(); }
    // One team per simulated warp; `neighbour_extra` > 0 plays a neighbour team (teams of 8 / 16 lanes share a warp) whose
    // loops run that many more trips, so the trips beyond this team's own count run too
    int warp_max(int v) const { return v + neighbour_extra; }
    static int neighbour_extra;
    double shfl(double v, int src) const {
        xd[lane] = v;
        team->yield();
        const double r = xd[src];
        team->yield();
        return r;
    }
    float shfl(float v, int src) const {
        xf[lane] = v;
        team->yield();
        const float r = xf[src];
        team->yield();
        return r;
    }
};

int HostCtx::neighbour_extra = 0;

struct Params {
    int max_it;
    double step, damping, tol;
    const double *lambdas;
};

template <typename T, class Cfg, bool SHFL, bool PIK>
void solve_all(const DevProblem<T> &P, const Params &prm, int B, const double *q0, const double *targets, double *q_out, int *success,
               int *iters, double *resid, double *e_first, double *J_first) {
    constexpr int TEAM = Cfg::TEAM;
    constexpr int EXTRA = 2;   // one scratch layout for all host runs (the buffers are simply unused by plain ik::dls)
    auto S = std::make_unique<CoopScratch<T, Cfg, EXTRA>>();
    double xd[32];
    float xf[32];
    T lam2[7];
    for (int l = 0; l < 7; ++l) lam2[l] = prm.lambdas ? (T)(prm.lambdas[l] * prm.lambdas[l]) : T(0);
    FiberTeam team;
    team.run(TEAM, [&](int lane) {
        const HostCtx cx{lane, &team, xd, xf};
        coop_init_scratch<T, Cfg, EXTRA>(cx, P, *S);
        for (int b = 0; b < B; ++b) {
            for (int k = lane; k < P.nq; k += TEAM) S->q[k] = (T)q0[(size_t)b * P.nq + k];
            for (int k = lane; k < P.tsz; k += TEAM) S->tg[k] = (T)targets[(size_t)b * P.tsz + k];
            cx.sync();
            int it = 0, ok = 0;
            T res = 0;
            while (it < prm.max_it) {
                res = coop_iteration<T, Cfg, SHFL, PIK, EXTRA>(cx, P, *S, (T)prm.step, (T)(prm.damping * prm.damping), lam2, (T)prm.tol);
                if (b == 0 && it == 0 && lane == 0) {
                    if (e_first) for (int i = 0; i < P.rows; ++i) e_first[i] = (double)S->e[i];
                    if (J_first) for (int i = 0; i < P.rows; ++i) for (int c = 0; c < P.nv; ++c) J_first[i * P.nv + c] = (double)S->Jt[c][i];
                }
                if (res < (T)prm.tol) { ok = 1; break; }
                ++it;
            }
            cx.sync();
            for (int k = lane; k < P.nq; k += TEAM) q_out[(size_t)b * P.nq + k] = (double)S->q[k];
            if (lane == 0) {
                success[b] = ok;
                iters[b] = it;
                resid[b] = (double)res;
            }
            cx.sync();
        }
    });
}

template <typename T, int CLS>
void solve_cls(const HostProblem &hp, int shfl, int pik, const Params &prm, int B, const double *q0, const double *targets, double *q_out,
               int *success, int *iters, double *resid, double *e_first, double *J_first) {
    using Cfg = typename CoopClass<CLS>::Cfg;
    auto P = std::make_unique<DevProblem<T>>();
    fill_dev_problem(hp, stacked_order(hp), used_frames(hp), *P);
    if (!P->coop_ok) throw std::runtime_error("problem exceeds the cooperative kernel's table capacities");
#define RUN(S_, P_) solve_all<T, Cfg, S_, P_>(*P, prm, B, q0, targets, q_out, success, iters, resid, e_first, J_first)
    if (pik) { if (shfl) RUN(true, true); else RUN(false, true); }
    else { if (shfl) RUN(true, false); else RUN(false, false); }
#undef RUN
}
}  // namespace

extern "C" void coop_set_neighbour_extra(int n) { HostCtx::neighbour_extra = n; }

extern "C" int coop_solve(const char *urdf, int free_flyer, int max_priority, int ntasks, const int *kind, const int *frame, const int *ref,
                          const int *type, const int *priority, const double *weights, const double *masks, int ncons,
                          const int *c_frame, const int *c_ref, const int *c_type, const double *lower, const double *upper, int f32,
                          int shfl, int pik, const double *lambdas, int max_it, double step, double damping, double tol, int B,
                          const double *q0, const double *targets, double *q_out, int *success, int *iters, double *resid,
                          double *e_first, double *J_first, int *cls_out) {
    try {
        HostProblem hp;
        hp.model = model_from_urdf(urdf, free_flyer != 0);
        if (lower && upper)
            for (int k = 0; k < hp.model.nq; ++k) { hp.model.lower[k] = lower[k]; hp.model.upper[k] = upper[k]; }
        hp.max_priority_level = max_priority;
        const double *w = weights, *mk = masks;
        for (int t = 0; t < ntasks; ++t) {
            HostTask ht;
            ht.kind = kind[t]; ht.frame = frame[t]; ht.ref = ref[t]; ht.type = type[t]; ht.priority = priority[t];
            if (ht.kind == IKB_TASK_FRAME) { ht.dim = ht.type == IKB_FULL ? 6 : 3; ht.target_size = 12; }
            else if (ht.kind == IKB_TASK_ALIGN_AXIS) { ht.dim = 1; ht.target_size = 3; }
            else if (ht.kind == IKB_TASK_POSTURE) { ht.dim = ht.type; ht.target_size = ht.type; ht.mask.assign(mk, mk + ht.type); mk += ht.type; }
            else { ht.dim = 3; ht.target_size = 3; ht.frame = ht.ref; }
            ht.weight.assign(w, w + ht.dim);
            w += ht.dim;
            hp.tasks.push_back(ht);
        }
        for (int c = 0; c < ncons; ++c) {
            HostConstraint hc;
            hc.frame = c_frame[c]; hc.ref = c_ref[c]; hc.type = c_type[c]; hc.dim = c_type[c] == IKB_FULL ? 6 : 3;
            hp.constraints.push_back(hc);
        }
        const int caps[3][3] = {{10, 8, 6}, {20, 24, 12}, {32, 36, 30}};
        int cls = -1;
        for (int c = 0; c < 3 && cls < 0; ++c)
            if (hp.model.njoints() <= caps[c][0] && hp.model.nv <= caps[c][1] && hp.rows() <= caps[c][2]) cls = c;
        if (cls < 0) return 2;
        if (cls == 2 && hp.model.njoints() <= 20 && hp.model.nv <= 24) cls = 3;   // the product's choice (ikb_solve.cu, coop_class)
        if (cls_out) *cls_out = cls;
        const Params prm{max_it, step, damping, tol, lambdas};
#define CALL(T_, C_) solve_cls<T_, C_>(hp, shfl, pik, prm, B, q0, targets, q_out, success, iters, resid, e_first, J_first)
        if (f32) { if (cls == 0) CALL(float, 0); else if (cls == 1) CALL(float, 1); else if (cls == 3) CALL(float, 3); else CALL(float, 2); }
        else { if (cls == 0) CALL(double, 0); else if (cls == 1) CALL(double, 1); else if (cls == 3) CALL(double, 3); else CALL(double, 2); }
#undef CALL
        return 0;
    } catch (const std::exception &e) {
        std::fprintf(stderr, "coop_harness: %s\n", e.what());
        return 1;
    }
}
