// lqgk_emul.cpp -- TEST INFRASTRUCTURE ONLY: runs the kernels' own step functions (lqg_b200/csrc/lqgk_core.h,
// lqgk_stages.h, lqgk_pack.h) sequentially on the CPU, exporting the same C ABI as liblqgk.so but on HOST
// pointers.  Lets `pytest -m "not gpu"` check the kernel mathematics (forward and adjoint) against the oracle
// without a GPU.  It is never loaded by the product path (lqg_b200 refuses anything but the CUDA library).
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/lqgk.h"
#include "../../lqg_b200/csrc/lqgk_core.h"
#include "../../lqg_b200/csrc/lqgk_entry.h"
#include "../../lqg_b200/csrc/lqgk_pack.h"
#include "../../lqg_b200/csrc/lqgk_stages.h"
#include "../../lqg_b200/csrc/lqgk_sdn.cuh"

using namespace lqgk;

namespace {

struct RecSink {
  float* row;  // rec[s][t][.]
  int rec;
  float* base;
  void put(int idx, float v) { row[idx] = v; }
  void commit(int t) { row = base + (size_t)(t + 1) * rec; }
};
struct SumSrc {
  const float* base;
  int sump;
  const float* row;
  void fetch(int t) { row = base + (size_t)t * sump; }
  float get(int idx) const { return row[idx]; }
};

template <class DM, class T>
int run(const Call& c) {
  const LqgkDims& d = *c.dims;
  const LqgkSpec *act = c.act, *dyn = c.dyn;
  const float* x_tm = c.x_tm;
  const T* ll_bar = (const T*)c.ll_bar;
  T *ll_out = (T*)c.ll_out, *L_out = (T*)c.L_out, *l_out = (T*)c.l_out, *H_out = (T*)c.H_out, *K_out = (T*)c.K_out;
  T *mu_out = (T*)c.mu_out, *Sig_out = (T*)c.Sig_out;
  const int mode = c.mode, S = d.S, N = d.N, Tn = d.T;
  const bool want_grad = mode == LQGK_MODE_VJP, has_dyn = dyn != nullptr;
  constexpr CLayout cl = DM::CL;
  const bool tv = spec_time_varying(*act, true) || (has_dyn && spec_time_varying(*dyn, false));
  if (!kernels_cover(c, tv, DM::N > 12)) return LQGK_E_UNSUPPORTED;
  const size_t Sc = S;
  const size_t tstride = tv ? (size_t)cl.total * Sc : 0;
  std::vector<double> cst((size_t)cl.total * Sc * (tv ? Tn : 1)), acc((size_t)cl.total * Sc, 0.0);
  PackArgs<T> pa{};
  pa.act = *act;
  if (has_dyn) pa.dyn = *dyn;
  pa.sigma0 = c.sigma0 ? *c.sigma0 : LqgkMat{nullptr, 0, 0};
  pa.x = DM::X; pa.b = DM::B; pa.u = DM::U; pa.y = DM::Y; pa.nT = Tn; pa.has_dyn = has_dyn;
  for (int t = 0; t < (tv ? Tn : 1); ++t)
    for (int s = 0; s < S; ++s) {
      WView out{cst.data() + (size_t)t * tstride + s, Sc};
      pack_sample<T>(pa, s, t, [&](int e) -> double& { return out(e); });
    }
  std::vector<double> Lw((size_t)Tn * DM::EL * Sc), Kw((size_t)Tn * DM::EK * Sc), Sw((size_t)Tn * DM::ES * Sc),
      Pw((size_t)Tn * DM::EP * Sc), Cw((size_t)Tn * DM::EC * Sc), Lbw((size_t)Tn * DM::EL * Sc),
      Kbw((size_t)Tn * DM::EK * Sc), lw((size_t)Tn * DM::U * Sc), Hw((size_t)Tn * DM::U * DM::U * Sc);
  using SR = CovSeqRev<DM>;
  constexpr int NC = CovC<DM>::n;
  const size_t adj = want_grad ? 1 : 0;
  std::vector<double> FUw(adj * Tn * SR::NSF * Sc), JSw(adj * Tn * SR::NJS * Sc), J0w(adj * DM::R * DM::D * Sc),
      SGBw(adj * Tn * SR::NSGB * Sc), SGBIw(adj * SR::NSGB * Sc), SFw(adj * Tn * SR::NSF * Sc), CTw(adj * Tn * NC * Sc);
  std::vector<double> lc(cl.total + 8), la(cl.total + 8);
  auto V = [&](std::vector<double>& v, int s) { return WView{v.data() + s, Sc}; };
  for (int s = 0; s < S; ++s) {
    GCst g{cst.data() + s, Sc, tstride};
    if (mode == LQGK_MODE_GAINS) {
      if (L_out) {
        lqr_fwd_body<DM, true>(g, WView{lc.data(), 1}, Tn, c.eps, V(Lw, s), false, V(Sw, s), V(lw, s), V(Hw, s));
        for (int t = 0; t < Tn; ++t) {
          for (int i = 0; i < DM::EL; ++i) L_out[((size_t)s * Tn + t) * DM::EL + i] = (T)Lw[((size_t)t * DM::EL + i) * Sc + s];
          if (l_out) for (int i = 0; i < DM::U; ++i) l_out[((size_t)s * Tn + t) * DM::U + i] = (T)lw[((size_t)t * DM::U + i) * Sc + s];
          if (H_out) for (int i = 0; i < DM::U * DM::U; ++i) H_out[((size_t)s * Tn + t) * DM::U * DM::U + i] = (T)Hw[((size_t)t * DM::U * DM::U + i) * Sc + s];
        }
      }
      if (K_out) {
        kf_fwd_body<DM>(g, WView{lc.data(), 1}, Tn, V(Kw, s), false, V(Pw, s));
        for (int t = 0; t < Tn; ++t)
          for (int i = 0; i < DM::EK; ++i) K_out[((size_t)s * Tn + t) * DM::EK + i] = (T)Kw[((size_t)t * DM::EK + i) * Sc + s];
      }
      continue;
    }
    lqr_fwd_body<DM, false>(g, WView{lc.data(), 1}, Tn, c.eps, V(Lw, s), want_grad, V(Sw, s), V(lw, s), V(Hw, s));
    kf_fwd_body<DM>(g, WView{lc.data(), 1}, Tn, V(Kw, s), want_grad, V(Pw, s));
  }
  if (mode == LQGK_MODE_GAINS) return LQGK_OK;
  std::vector<float> rec((size_t)Sc * Tn * DM::REC, 0.f), sums((size_t)Sc * Tn * DM::SUMP, 0.f),
      hist(want_grad ? (size_t)Sc * Tn * N * DM::R : 0);
  for (int s = 0; s < S; ++s) {
    GCst g{cst.data() + s, Sc, tstride};
    RecSink sink{rec.data() + (size_t)s * Tn * DM::REC, DM::REC, rec.data() + (size_t)s * Tn * DM::REC};
    if (mode == LQGK_MODE_MOMENTS)   // (what k_cov_moments does: the record plus the full predictive joint covariance of every step)
      cov_fwd_body<DM>(g, WView{lc.data(), 1}, Tn, V(Lw, s), V(Kw, s), false, V(Cw, s), V(FUw, s), V(JSw, s), V(J0w, s), sink,
                       [&](int t, int e, double v) { if (Sig_out) Sig_out[((size_t)s * Tn + t) * (DM::N * DM::N) + e] = (T)v; });
    else
      cov_fwd_body<DM>(g, WView{lc.data(), 1}, Tn, V(Lw, s), V(Kw, s), want_grad, V(Cw, s), V(FUw, s), V(JSw, s), V(J0w, s), sink);
  }
  if (mode == LQGK_MODE_MOMENTS) {   // (k_trial_moments)
    if (mu_out)
      for (int s = 0; s < S; ++s)
        for (int i = 0; i < N; ++i) {
          const float* xs = x_tm + (size_t)s * d.x_sample_stride;
          float c[DM::R] = {0}, mu[DM::N];
          for (int t = 0; t < Tn; ++t) {
            Trial<DM>::template moments<float>(rec.data() + ((size_t)s * Tn + t) * DM::REC, xs + ((size_t)t * N + i) * DM::D,
                                               xs + ((size_t)(t + 1) * N + i) * DM::D, c, mu);
            for (int k = 0; k < DM::N; ++k) mu_out[(((size_t)s * N + i) * Tn + t) * DM::N + k] = (T)mu[k];
          }
        }
    return LQGK_OK;
  }
  // the library stores these adjoint linearisation points in FP32 (lin_t in lqgk_kernels.cuh): mirror the rounding
  for (auto& v : FUw) v = (double)(float)v;
  for (auto& v : JSw) v = (double)(float)v;
  using TR = Trial<DM>;
  constexpr int D = DM::D, R = DM::R;
  const float* x_all = x_tm;
  for (int s = 0; s < S; ++s)
    for (int i = 0; i < N; ++i) {
      const float* x_tm = x_all + (size_t)s * d.x_sample_stride;
      float c[R] = {0};
      double ll = 0.0;
      for (int t = 0; t < Tn; ++t) {
        const float* r = rec.data() + ((size_t)s * Tn + t) * DM::REC;
        if (want_grad) std::memcpy(&hist[(((size_t)s * Tn + t) * N + i) * R], c, sizeof(float) * R);
        ll += (double)TR::template fwd<float>(r, x_tm + ((size_t)t * N + i) * D, x_tm + ((size_t)(t + 1) * N + i) * D, c);
      }
      ll_out[(size_t)s * N + i] = (T)ll;
    }
  if (!want_grad) return LQGK_OK;
  for (int s = 0; s < S; ++s) {
    const float* x_tm = x_all + (size_t)s * d.x_sample_stride;
    double sw = 0.0;
    for (int i = 0; i < N; ++i) {
      float w = ll_bar ? (float)ll_bar[(size_t)s * N + i] : 1.f;
      sw += w;
      float cb[R] = {0};
      for (int t = Tn - 1; t >= 0; --t) {
        const float* r = rec.data() + ((size_t)s * Tn + t) * DM::REC;
        const float* c = &hist[(((size_t)s * Tn + t) * N + i) * R];
        const float* x0 = x_tm + ((size_t)t * N + i) * D;
        const float* x1 = x_tm + ((size_t)(t + 1) * N + i) * D;
        float e[D], v[D], wv[D], neb[D], cbn[R];
        TR::template rev<float>(r, x0, x1, c, w, cb, e, v, wv, neb, cbn);
        float* sm = sums.data() + ((size_t)s * Tn + t) * DM::SUMP;
        static_for<0, DM::NSUM>([&](auto I) {
          sm[decltype(I)::value] = TR::template sum_acc<decltype(I)::value, float>(sm[decltype(I)::value], cb, neb, x0, c, e, v, wv);
        });
        for (int j = 0; j < R; ++j) cb[j] = cbn[j];
      }
    }
    GCst g{cst.data() + s, Sc, 0};
    WView ga{acc.data() + s, Sc};
    SumSrc src{sums.data() + (size_t)s * Tn * DM::SUMP, DM::SUMP, nullptr};
    {
      std::vector<double> sc(SR::SC_N + 8);
      cov_seq_rev_body<DM>(Tn, sw, V(FUw, s), V(JSw, s), V(J0w, s), src, WView{sc.data(), 1}, V(SGBw, s), V(SGBIw, s), V(SFw, s));
      for (size_t e = s; e < SGBw.size(); e += Sc) SGBw[e] = (double)(float)SGBw[e];   // (FP32 storage, as in the library)
      for (size_t e = s; e < SFw.size(); e += Sc) SFw[e] = (double)(float)SFw[e];
      load_consts<CovC<DM>>(g.at(0), WView{lc.data(), 1}, CovC<DM>::NSEG);
      auto ct = [&](int t, int e, double v) { CTw[((size_t)t * NC + e) * Sc + s] = v; };
      cov_contrib_body<DM, 0>(WView{lc.data(), 1}, 0, Tn, V(Lw, s), V(Kw, s), V(Cw, s), V(SGBw, s), V(SGBIw, s), V(SFw, s), src,
                              ct, V(Lbw, s), V(Kbw, s));
      cov_contrib_body<DM, 1>(WView{lc.data(), 1}, 0, Tn, V(Lw, s), V(Kw, s), V(Cw, s), V(SGBw, s), V(SGBIw, s), V(SFw, s), src,
                              ct, V(Lbw, s), V(Kbw, s));
      for (int e = 0; e < NC; ++e) la[e] = 0.0;               // time reduction of the per-step contributions
      for (int t = 0; t < Tn; ++t)
        for (int e = 0; e < NC; ++e) la[e] += CTw[((size_t)t * NC + e) * Sc + s];
      flush_acc<CovC<DM>>(ga, WView{la.data(), 1}, CovC<DM>::NSEG);
    }
    kf_rev_body<DM>(g, WView{lc.data(), 1}, WView{la.data(), 1}, Tn, V(Pw, s), V(Kbw, s), ga);
    lqr_rev_body<DM>(g, WView{lc.data(), 1}, WView{la.data(), 1}, Tn, c.eps, V(Lw, s), V(Sw, s), V(Lbw, s), ga);
    UnpackArgs<T> ua{};
    ua.act = *act; ua.dyn = *dyn; ua.sigma0 = pa.sigma0;
    if (c.gact) ua.gact = *c.gact;
    if (c.gdyn) ua.gdyn = *c.gdyn;
    if (c.gsig0) ua.gsigma0 = *c.gsig0;
    ua.x = DM::X; ua.b = DM::B; ua.u = DM::U; ua.y = DM::Y;
    WView cv{cst.data() + s, Sc};
    unpack_sample<T>(ua, s, [&](int e) { return (double)ga(e); }, [&](int e) { return (double)cv(e); });
  }
  return LQGK_OK;
}

template <class T>
int dispatch(const Call& c) {
  if (int rc = validate(c)) return rc;
  return visit_tuple<Tuples::compiled>(call_key(*c.dims, c.mode), LQGK_E_UNSUPPORTED, [&](auto dm, auto) { return run<decltype(dm), T>(c); });
}

template <class T>
int pack_obs_host(int32_t N, int32_t T1, int32_t d, const T* x, float* x_tm) {
  if (int rc = check_pack_obs(N, T1, d, x, x_tm)) return rc;
  for (int i = 0; i < N; ++i)
    for (int t = 0; t < T1; ++t)
      for (int k = 0; k < d; ++k) x_tm[((size_t)t * N + i) * d + k] = (float)x[((size_t)i * T1 + t) * d + k];
  return LQGK_OK;
}
template <class T>
int sdn_loglik_host(const LqgkDims* d, const LqgkSpec* act, const LqgkSpec* dyn, const LqgkSdnNoise* nz, const T* L, const T* K,
                    const float* x_tm, T* ll_out) {
  SdnLikArgs a;
  if (int rc = sdn_lik_args(d, act, dyn, nz, L, K, x_tm, ll_out, a)) return rc;
  return visit_tuple<Tuples::small_and_fp64_only>(full_key(*d), LQGK_E_UNSUPPORTED, [&](auto dm, auto) {
    for (int s = 0; s < a.S; ++s)
      for (int i = 0; i < a.N; ++i) ll_out[(size_t)s * a.N + i] = (T)SdnLik<decltype(dm)>::template trial<T>(a, s, i);
    return LQGK_OK;
  });
}
int sdn_gains_host(const LqgkSdnDims* d, const LqgkSdnSpec* sp, double* L_out, double* K_out, double* cost_out, int filter_form) {
  SdnArgs a;
  if (int rc = sdn_gains_args(d, sp, L_out, K_out, cost_out, filter_form, a)) return rc;
  return visit_tuple<Tuples::small>(TupleKey{ANY, d->b, d->u, d->y, ANY}, LQGK_E_UNSUPPORTED, [&](auto dm, auto) {
    for (int s = 0; s < a.S; ++s) {
      const double c = Sdn<decltype(dm)>::solve(a, s);
      if (cost_out) cost_out[s] = c;
    }
    return LQGK_OK;
  });
}
}  // namespace

extern "C" {
int lqgk_sdn_gains_f64(const LqgkSdnDims* d, const LqgkSdnSpec* sp, double* L_out, double* K_out, double* cost_out, void*) {
  return sdn_gains_host(d, sp, L_out, K_out, cost_out, 0);
}
int lqgk_sdn_gains_filter_f64(const LqgkSdnDims* d, const LqgkSdnSpec* sp, double* L_out, double* K_out, double* cost_out, void*) {
  return sdn_gains_host(d, sp, L_out, K_out, cost_out, 1);
}
int lqgk_sdn_loglik_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkSdnNoise* noise, const double* L,
                        const double* K, const float* x_tm, double* ll_out, void*) {
  return sdn_loglik_host<double>(dims, actor, dynamics, noise, L, K, x_tm, ll_out);
}
int lqgk_lqr_backward_f64(const LqgkDims* dims, const LqgkSpec* actor, double eps, double* L_out, double* l_out,
                          double* H_out, void*, size_t, void*) {
  Call c;
  c.mode = LQGK_MODE_GAINS; c.dims = dims; c.act = actor; c.eps = eps; c.L_out = L_out; c.l_out = l_out; c.H_out = H_out;
  return dispatch<double>(c);
}
int lqgk_kf_forward_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, double* K_out, void*,
                        size_t, void*) {
  Call c;
  c.mode = LQGK_MODE_GAINS; c.dims = dims; c.act = actor; c.sigma0 = sigma0; c.K_out = K_out;
  return dispatch<double>(c);
}
int lqgk_loglik_fwd_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0,
                        const float* x_tm, double* ll_out, void*, size_t, void*) {
  Call c;
  c.mode = LQGK_MODE_FWD; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.ll_out = ll_out;
  return dispatch<double>(c);
}
int lqgk_loglik_vjp_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0,
                        const float* x_tm, const double* ll_bar, double* ll_out, const LqgkSpecGrad* ga,
                        const LqgkSpecGrad* gd, const LqgkMatGrad* gs, void*, size_t, void*) {
  Call c;
  c.mode = LQGK_MODE_VJP; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.ll_bar = ll_bar;
  c.ll_out = ll_out; c.gact = ga; c.gdyn = gd; c.gsig0 = gs;
  return dispatch<double>(c);
}
int lqgk_loglik_fwd_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0,
                        const float* x_tm, float* ll_out, void*, size_t, void*) {
  Call c;
  c.mode = LQGK_MODE_FWD; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.ll_out = ll_out;
  return dispatch<float>(c);
}
int lqgk_loglik_vjp_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0,
                        const float* x_tm, const float* ll_bar, float* ll_out, const LqgkSpecGrad* ga,
                        const LqgkSpecGrad* gd, const LqgkMatGrad* gs, void*, size_t, void*) {
  Call c;
  c.mode = LQGK_MODE_VJP; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.ll_bar = ll_bar;
  c.ll_out = ll_out; c.gact = ga; c.gdyn = gd; c.gsig0 = gs;
  return dispatch<float>(c);
}
int lqgk_moments_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0, const float* x_tm,
                     double* mu_out, double* Sigma_out, void*, size_t, void*) {
  Call c;
  c.mode = LQGK_MODE_MOMENTS; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.mu_out = mu_out;
  c.Sig_out = Sigma_out;
  return dispatch<double>(c);
}
int lqgk_moments_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0, const float* x_tm,
                     float* mu_out, float* Sigma_out, void*, size_t, void*) {
  Call c;
  c.mode = LQGK_MODE_MOMENTS; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.mu_out = mu_out;
  c.Sig_out = Sigma_out;
  return dispatch<float>(c);
}
int lqgk_pack_obs_f32(int32_t N, int32_t T1, int32_t d, const float* x, float* x_tm, void*) { return pack_obs_host(N, T1, d, x, x_tm); }
int lqgk_pack_obs_f64(int32_t N, int32_t T1, int32_t d, const double* x, float* x_tm, void*) { return pack_obs_host(N, T1, d, x, x_tm); }
int lqgk_last_launch_count(void) { return 0; }
const char* lqgk_version(void) { return "lqgk-emul (CPU test harness, not a product path)"; }
}
