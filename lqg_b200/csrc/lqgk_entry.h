// lqgk_entry.h -- what an entry point does before it computes, written once for liblqgk.so (lqgk_api.cu) and its host build
// (tests/emul/lqgk_emul.cpp): the argument checks, the SDN argument builders and the dimension dispatch.  Host code only.
#pragma once
#include <initializer_list>

#include "../../include/lqgk.h"
#include "lqgk_core.h"
#include "lqgk_dims.h"
#include "lqgk_sdn.cuh"

struct CUstream_st;   // (cudaStream_t is CUstream_st*)

namespace lqgk {

// The arguments of a gains, likelihood, adjoint or moments call; an entry point sets the fields of its kind.
struct Call {
  const LqgkDims* dims = nullptr;
  const LqgkSpec *act = nullptr, *dyn = nullptr;
  const LqgkMat* sigma0 = nullptr;
  const float* x_tm = nullptr;
  const void* ll_bar = nullptr;
  const void *L_bar = nullptr, *K_bar = nullptr;   // cotangents of the gains (gains adjoint)
  const LqgkSpecGrad *gact = nullptr, *gdyn = nullptr;
  const LqgkMatGrad* gsig0 = nullptr;
  void *ll_out = nullptr, *L_out = nullptr, *l_out = nullptr, *H_out = nullptr, *K_out = nullptr, *mu_out = nullptr, *Sig_out = nullptr;
  double eps = 1e-8;
  int mode = LQGK_MODE_FWD;
  void* ws = nullptr;
  size_t ws_bytes = 0;
  CUstream_st* stream = nullptr;
};

// LQGK_E_INVALID unless every matrix is given; with `time_invariant`, LQGK_E_UNSUPPORTED for a time-varying one.
inline int need(std::initializer_list<const LqgkMat*> mats, bool time_invariant = false) {
  for (auto m : mats) {
    if (!m->ptr) return LQGK_E_INVALID;
    if (time_invariant && m->time_stride != 0) return LQGK_E_UNSUPPORTED;
  }
  return LQGK_OK;
}
// the matrices the closed loop of the simulator and of the SDN likelihood reads
inline int need_closed_loop(const LqgkSpec& act, const LqgkSpec& dyn, bool time_invariant) {
  return need({&act.A, &act.B, &act.F, &dyn.A, &dyn.B, &dyn.F, &dyn.V, &dyn.W}, time_invariant);
}

// the modes that run the gain sweeps alone (no observations, no dynamics spec)
inline bool gains_mode(int mode) { return mode == LQGK_MODE_GAINS || mode == LQGK_MODE_GAINS_VJP; }

inline int validate(const Call& c) {
  if (!c.dims || !c.act) return LQGK_E_INVALID;
  const LqgkDims& d = *c.dims;
  if (d.S <= 0 || d.T <= 0 || d.x <= 0 || d.b <= 0 || d.u <= 0 || d.y <= 0) return LQGK_E_INVALID;
  if (!c.act->A.ptr || !c.act->B.ptr) return LQGK_E_INVALID;
  if (c.mode == LQGK_MODE_GAINS && !c.L_out && !c.K_out) return LQGK_E_INVALID;
  if (c.mode == LQGK_MODE_GAINS_VJP) {
    if (!c.L_bar && !c.K_bar) return LQGK_E_INVALID;
    const LqgkSpec& a = *c.act;
    if (need({&a.F, &a.V, &a.W, &a.Q, &a.R})) return LQGK_E_INVALID;
    if (a.P.ptr) return LQGK_E_UNSUPPORTED;   // the Riccati adjoint has no cross-cost term
  }
  if (!gains_mode(c.mode)) {
    if (d.N <= 0 || d.d <= 0 || d.d > d.x) return LQGK_E_INVALID;
    if (!c.dyn || !c.x_tm) return LQGK_E_INVALID;
    if (c.mode == LQGK_MODE_MOMENTS ? (!c.mu_out && !c.Sig_out) : !c.ll_out) return LQGK_E_INVALID;
    const LqgkSpec &a = *c.act, &dy = *c.dyn;
    if (need({&a.F, &a.V, &a.W, &a.Q, &a.R, &dy.A, &dy.B, &dy.F, &dy.V, &dy.W})) return LQGK_E_INVALID;
    if (((uintptr_t)c.x_tm % 16) != 0) return LQGK_E_INVALID;
    // per-sample data sets: every sample's block must keep the alignment of the kernels' observation accesses (one d-float
    // vector per trial: 16 bytes when d % 4 == 0, 8 when d % 2 == 0, else scalar loads)
    const size_t xalign = d.d % 4 == 0 ? 16 : (d.d % 2 == 0 ? 8 : 4);
    if (d.x_sample_stride < 0 || (d.x_sample_stride * sizeof(float)) % xalign != 0) return LQGK_E_INVALID;
  }
  return LQGK_OK;
}

inline bool spec_time_varying(const LqgkSpec& s, bool actor) {
  const LqgkMat* m[] = {&s.A, &s.B, &s.F, &s.V, &s.W, &s.Q, &s.R, &s.q, &s.r, &s.P};
  int n = actor ? 10 : 5;
  for (int i = 0; i < n; ++i)
    if (m[i]->ptr && m[i]->time_stride != 0) return true;
  return false;
}
// What the kernels of a tuple leave out (tv: a time-varying spec; big: joint dim > 12): the adjoints of a time-varying spec,
// and for large systems time-varying specs and the predictive moments.
inline bool kernels_cover(const Call& c, bool tv, bool big) {
  if (tv && (c.mode == LQGK_MODE_VJP || c.mode == LQGK_MODE_GAINS_VJP)) return false;
  return !(big && (tv || c.mode == LQGK_MODE_MOMENTS));
}

// The gains adjoint (lqgk_gains_vjp_*): `base` receives the actor spec without its affine terms q, r, qf, which the gains do
// not depend on, so that neither their presence nor a time axis of theirs matters.
inline Call gains_vjp_call(const LqgkDims* dims, const LqgkSpec* act, const LqgkMat* sigma0, double eps, const void* L_bar,
                           const void* K_bar, const LqgkSpecGrad* ga, const LqgkMatGrad* gs, LqgkSpec& base) {
  Call c;
  c.mode = LQGK_MODE_GAINS_VJP; c.dims = dims; c.sigma0 = sigma0; c.eps = eps; c.L_bar = L_bar; c.K_bar = K_bar; c.gact = ga;
  c.gsig0 = gs;
  if (act) {
    base = *act;
    base.q = base.r = base.qf = LqgkMat{nullptr, 0, 0};
    c.act = &base;
  }
  return c;
}

inline int check_pack_obs(int32_t N, int32_t T1, int32_t d, const void* x, const float* x_tm) {
  return N <= 0 || T1 <= 0 || d <= 0 || !x || !x_tm ? LQGK_E_INVALID : LQGK_OK;
}

// The multiplicative-noise terms of the SDN simulator and likelihood (none when nz is null).
inline int check_noise(const LqgkSdnNoise* nz) {
  if (!nz) return LQGK_OK;
  if (nz->nc < 0 || nz->nd < 0 || nz->nc > SDN_MAX_TERMS || nz->nd > SDN_MAX_TERMS) return LQGK_E_INVALID;
  if ((nz->nc > 0 && !nz->C.ptr) || (nz->nd > 0 && !nz->D.ptr)) return LQGK_E_INVALID;
  return LQGK_OK;
}

inline int sdn_gains_args(const LqgkSdnDims* d, const LqgkSdnSpec* sp, double* L_out, double* K_out, double* cost_out,
                          int filter_form, SdnArgs& a) {
  if (!d || !sp || !L_out || !K_out) return LQGK_E_INVALID;
  if (d->S <= 0 || d->T <= 0 || d->b <= 0 || d->u <= 0 || d->y <= 0 || d->nc < 0 || d->nd < 0 || d->sweeps < 0) return LQGK_E_INVALID;
  if (need({&sp->A, &sp->B, &sp->H, &sp->Q, &sp->R, &sp->Om_xi, &sp->Om_omega, &sp->Sigma1, &sp->xhat1})) return LQGK_E_INVALID;
  if ((d->nc > 0 && !sp->C.ptr) || (d->nd > 0 && !sp->D.ptr)) return LQGK_E_INVALID;
  a = SdnArgs{};
  auto set = [](const double*& p, long long& sample_stride, const LqgkMat& m) { p = (const double*)m.ptr; sample_stride = m.sample_stride; };
  set(a.A, a.sA, sp->A); set(a.B, a.sB, sp->B); set(a.H, a.sH, sp->H); set(a.C, a.sC, sp->C); set(a.D, a.sD, sp->D);
  set(a.Q, a.sQ, sp->Q); set(a.R, a.sR, sp->R); set(a.Qf, a.sQf, sp->Qf.ptr ? sp->Qf : sp->Q); set(a.Omxi, a.sOmxi, sp->Om_xi);
  set(a.Omom, a.sOmom, sp->Om_omega); set(a.Sig1, a.sSig1, sp->Sigma1); set(a.xh1, a.sxh1, sp->xhat1);
  a.S = d->S; a.T = d->T; a.nc = d->nc; a.nd = d->nd; a.sweeps = d->sweeps;
  a.L = L_out; a.K = K_out; a.cost = cost_out; a.filter_form = filter_form;
  return LQGK_OK;
}

inline int sdn_lik_args(const LqgkDims* d, const LqgkSpec* act, const LqgkSpec* dyn, const LqgkSdnNoise* nz, const void* L,
                        const void* K, const float* x_tm, void* ll_out, SdnLikArgs& a) {
  if (!d || !act || !dyn || !L || !K || !x_tm || !ll_out) return LQGK_E_INVALID;
  if (d->S <= 0 || d->N <= 0 || d->T <= 0 || d->d <= 0 || d->d > d->x || d->x_sample_stride < 0) return LQGK_E_INVALID;
  if (int rc = need_closed_loop(*act, *dyn, true)) return rc;
  if (int rc = check_noise(nz)) return rc;
  a = SdnLikArgs{};
  a.act = *act; a.dyn = *dyn; a.L = L; a.K = K; a.x_tm = x_tm; a.x_sample_stride = d->x_sample_stride; a.ll_out = ll_out;
  a.S = d->S; a.N = d->N; a.T = d->T;
  if (nz) { a.C = nz->C; a.D = nz->D; a.nc = nz->nc; a.nd = nz->nd; }
  return LQGK_OK;
}

// ------------------------------------------------------------------------------------------------- dimension dispatch
// A call's key into the compiled tuples: a field set to ANY matches every tuple.
constexpr int ANY = -1;
struct TupleKey {
  int x, b, u, y, d;
};
inline TupleKey full_key(const LqgkDims& d) { return {d.x, d.b, d.u, d.y, d.d}; }
// the gains sweeps do not read the observations: their d is any tuple's
inline TupleKey call_key(const LqgkDims& d, int mode) { return {d.x, d.b, d.u, d.y, gains_mode(mode) ? ANY : d.d}; }

enum class Tuples {
  compiled,              // every line of LQGK_FOR_EACH_DIMS
  small,                 // those of joint dim <= 12 (the SDN gains)
  small_and_fp64_only,   // those, then the lines of LQGK_FOR_EACH_FP64_ONLY_DIMS (the SDN / all-FP64 likelihood)
};

// f(Dims<X, B, U, Y, D>{}, fp64_only) for the first tuple of SET that `key` matches (fp64_only: std::true_type for a line of
// LQGK_FOR_EACH_FP64_ONLY_DIMS), `none` when there is none.  f is instantiated for the tuples of SET only.
template <Tuples SET, class R, class F>
R visit_tuple(const TupleKey& key, R none, F&& f) {
  auto hit = [&](int X, int B, int U, int Y, int D) {
    return (key.x == ANY || key.x == X) && (key.b == ANY || key.b == B) && (key.u == ANY || key.u == U) &&
           (key.y == ANY || key.y == Y) && (key.d == ANY || key.d == D);
  };
#define LQGK_VISIT(X, B, U, Y, D)                                              \
  if constexpr (SET == Tuples::compiled || X + B <= 12) {                      \
    if (hit(X, B, U, Y, D)) return f(Dims<X, B, U, Y, D>{}, std::false_type{}); \
  }
  LQGK_FOR_EACH_DIMS(LQGK_VISIT)
#undef LQGK_VISIT
#define LQGK_VISIT(X, B, U, Y, D)                                             \
  if constexpr (SET == Tuples::small_and_fp64_only) {                         \
    if (hit(X, B, U, Y, D)) return f(Dims<X, B, U, Y, D>{}, std::true_type{}); \
  }
  LQGK_FOR_EACH_FP64_ONLY_DIMS(LQGK_VISIT)
#undef LQGK_VISIT
  return none;
}

}  // namespace lqgk
