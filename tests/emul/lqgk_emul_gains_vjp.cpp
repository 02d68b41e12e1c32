// lqgk_emul_gains_vjp.cpp -- TEST INFRASTRUCTURE ONLY: the host build of every entry point (lqgk_emul.cpp) plus the adjoint of
// the gain sweeps, lqgk_gains_vjp_*, from the kernels' own step functions (lqr_fwd_body / kf_fwd_body keeping S_t / P_t, then
// lqr_rev_body / kf_rev_body and unpack_sample), run sequentially on the CPU on HOST pointers.  Built into
// tests/emul/liblqgk_emul_gains.so; lets `pytest -m "not gpu"` check the gains adjoint against the oracle without a GPU.
#include "lqgk_emul.cpp"

namespace {

// What Chunk / run<DM, T> in lqgk_run.cuh do for LQGK_MODE_GAINS_VJP, one sample after the other.
template <class DM, class T>
int run_gains_vjp(const Call& c) {
  const LqgkDims& d = *c.dims;
  const int S = d.S, Tn = d.T;
  if (!kernels_cover(c, spec_time_varying(*c.act, true), DM::N > 12)) return LQGK_E_UNSUPPORTED;
  constexpr CLayout cl = DM::CL;
  const size_t Sc = S;
  std::vector<double> cst((size_t)cl.total * Sc), acc((size_t)cl.total * Sc, 0.0), lc(cl.total + 8), la(cl.total + 8);
  std::vector<double> Lw((size_t)Tn * DM::EL * Sc), Kw((size_t)Tn * DM::EK * Sc), Sw((size_t)Tn * DM::ES * Sc),
      Pw((size_t)Tn * DM::EP * Sc), Lbw((size_t)Tn * DM::EL * Sc), Kbw((size_t)Tn * DM::EK * Sc), lw((size_t)Tn * DM::U * Sc),
      Hw((size_t)Tn * DM::U * DM::U * Sc);
  auto V = [&](std::vector<double>& v, int s) { return WView{v.data() + s, Sc}; };
  PackArgs<T> pa{};
  pa.act = *c.act;
  pa.sigma0 = c.sigma0 ? *c.sigma0 : LqgkMat{nullptr, 0, 0};
  pa.x = DM::X; pa.b = DM::B; pa.u = DM::U; pa.y = DM::Y; pa.nT = Tn; pa.has_dyn = 0;
  const T *L_bar = (const T*)c.L_bar, *K_bar = (const T*)c.K_bar;
  for (int s = 0; s < S; ++s) {
    WView out{cst.data() + s, Sc};
    pack_sample<T>(pa, s, 0, [&](int e) -> double& { return out(e); });
    GCst g{cst.data() + s, Sc, 0};
    WView ga{acc.data() + s, Sc};
    if (L_bar) {
      lqr_fwd_body<DM, false>(g, WView{lc.data(), 1}, Tn, c.eps, V(Lw, s), true, V(Sw, s), V(lw, s), V(Hw, s));
      for (int t = 0; t < Tn; ++t)
        for (int i = 0; i < DM::EL; ++i) Lbw[((size_t)t * DM::EL + i) * Sc + s] = (double)L_bar[((size_t)s * Tn + t) * DM::EL + i];
      lqr_rev_body<DM>(g, WView{lc.data(), 1}, WView{la.data(), 1}, Tn, c.eps, V(Lw, s), V(Sw, s), V(Lbw, s), ga);
    }
    if (K_bar) {
      kf_fwd_body<DM>(g, WView{lc.data(), 1}, Tn, V(Kw, s), true, V(Pw, s));
      for (int t = 0; t < Tn; ++t)
        for (int i = 0; i < DM::EK; ++i) Kbw[((size_t)t * DM::EK + i) * Sc + s] = (double)K_bar[((size_t)s * Tn + t) * DM::EK + i];
      kf_rev_body<DM>(g, WView{lc.data(), 1}, WView{la.data(), 1}, Tn, V(Pw, s), V(Kbw, s), ga);
    }
    UnpackArgs<T> ua{};
    ua.act = *c.act; ua.sigma0 = pa.sigma0;
    if (c.gact) ua.gact = *c.gact;
    if (c.gsig0) ua.gsigma0 = *c.gsig0;
    ua.x = DM::X; ua.b = DM::B; ua.u = DM::U; ua.y = DM::Y;
    unpack_sample<T, false>(ua, s, [&](int e) { return (double)ga(e); }, [&](int e) { return (double)out(e); });
  }
  return LQGK_OK;
}

template <class T>
int gains_vjp_host(const Call& c) {
  if (int rc = validate(c)) return rc;
  return visit_tuple<Tuples::compiled>(call_key(*c.dims, c.mode), LQGK_E_UNSUPPORTED,
                                       [&](auto dm, auto) { return run_gains_vjp<decltype(dm), T>(c); });
}

}  // namespace

extern "C" {
int lqgk_gains_vjp_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, double eps, const double* L_bar,
                       const double* K_bar, const LqgkSpecGrad* ga, const LqgkMatGrad* gs, void*, size_t, void*) {
  LqgkSpec base;
  return gains_vjp_host<double>(gains_vjp_call(dims, actor, sigma0, eps, L_bar, K_bar, ga, gs, base));
}
int lqgk_gains_vjp_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, double eps, const float* L_bar,
                       const float* K_bar, const LqgkSpecGrad* ga, const LqgkMatGrad* gs, void*, size_t, void*) {
  LqgkSpec base;
  return gains_vjp_host<float>(gains_vjp_call(dims, actor, sigma0, eps, L_bar, K_bar, ga, gs, base));
}
}
