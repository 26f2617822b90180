// TEST-ONLY: the generated body of a plugin specialisation with FrameConstraints (-DIKB_PLUGIN_HEADER="...",
// -DIKB_PLUGIN_STRUCT=...) driven on the CPU by spec_harness.cpp's loop, exported as h_spec_plugin_{d,f,pd}, and one
// evaluation with the constraint Jacobian and the projected step, h_spec_plugin_ceval.  Never linked into libikb200.so.
#include "spec_harness.cpp"
#include IKB_PLUGIN_HEADER

using SP = IKB_PLUGIN_STRUCT;

extern "C" int h_spec_plugin_d(const double *lo, const double *hi, const double *w, const double *mk, const double *q0, const double *tg,
                               int mi, double st, double da, double tol, double *q, int *it, double *res, double *e0) {
    return spec_solve<SP, double>(lo, hi, w, mk, q0, tg, mi, st, da, tol, q, it, res, e0);
}
extern "C" int h_spec_plugin_f(const double *lo, const double *hi, const double *w, const double *mk, const double *q0, const double *tg,
                               int mi, double st, double da, double tol, double *q, int *it, double *res, double *e0) {
    return spec_solve<SP, float>(lo, hi, w, mk, q0, tg, mi, st, da, tol, q, it, res, e0);
}
extern "C" int h_spec_plugin_pd(const double *lo, const double *hi, const double *w, const double *mk, const double *q0, const double *tg,
                                int mi, double st, double da, double tol, double *q, int *it, double *res, double *e0) {
    return spec_solve<SP, double>(lo, hi, w, mk, q0, tg, mi, st, da, tol, q, it, res, e0, true);
}

// One evaluation at q0: weighted e[M], the dense weighted task Jacobian J[M][NV] (from the task slots), the dense
// constraint Jacobian Jc[MC][NV] (from the constraint slots), and dq = step_direction(y), i.e. -(I - P) J^T y.  Returns the
// rank project() finds for Jc.
extern "C" int h_spec_plugin_ceval(const double *weight, const double *q0, const double *targets, const double *y_in, double *e_out,
                                   double *J_out, double *Jc_out, double *dq_out) {
    constexpr int NV = SP::NV, M = SP::M;
    SpecConsts<double, SP::NQ, M> c{};
    for (int i = 0; i < M; ++i) {
        c.weight[i] = weight[i];
        c.mask[i] = 1.0;
    }
    std::vector<double> bufJ(SP::NSLOT), bufT(targets, targets + SP::TSZ), bufE(M);
    const Strip<double, 1> sJ{bufJ.data()}, sT{bufT.data()}, sE{bufE.data()};
    auto evaluate = [&]() {
        for (int role = 0; role < SP::NWARPS; ++role) {
            double q[SP::NQL];
            SP::load_q(role, q0, 1LL, q);
            SP::evaluate(role, q, sT, c, sJ, sE);
        }
    };
    evaluate();
    for (int i = 0; i < M; ++i) e_out[i] = bufE[i];
    for (int i = 0; i < M * NV; ++i) J_out[i] = 0;
    for (int k = 0; k < SP::CSLOT; ++k) J_out[SP::slot_rc()[2 * k] * NV + SP::slot_rc()[2 * k + 1]] = bufJ[k];
    for (int i = 0; i < SP::MC * NV; ++i) Jc_out[i] = 0;
    for (int r = 0; r < SP::MC; ++r)
        for (int u = 0; u < SP::NU; ++u) Jc_out[r * NV + SP::con_cols()[u]] = bufJ[SP::CSLOT + r * SP::NU + u];
    double y[M];
    for (int i = 0; i < M; ++i) y[i] = y_in[i];
    double dq[NV];
    SP::step_direction(sJ, y, dq);
    for (int k = 0; k < NV; ++k) dq_out[k] = dq[k];
    evaluate();   // (project() factorised Jc in place)
    double d0[NV] = {};
    return SP::project(sJ, d0);
}
