// lqgk_pack.h -- generic (run-time dimension) boundary code: base matrices <-> derived constants.
//
// pack_sample   : reads the caller's base matrices (any strides, f32/f64) of one sample at one time step and
//                 writes the block of derived constants (CLayout, FP64, sample-minor) the kernels consume.
// unpack_sample : chains the accumulated cotangents of the derived constants back to the 12 base matrices
//                 (oracle/adjoint_np.py: derived_to_base) and stores them in the caller's gradient buffers.
// Both run once per sample (not per time step) and are therefore written for clarity, not speed.
#pragma once
#include "../../include/lqgk.h"
#include "lqgk_core.h"

namespace lqgk {

template <class T>
LQGK_HD double mat_at(const LqgkMat& m, int s, int t, int idx) {
  return (double)((const T*)m.ptr)[(int64_t)s * m.sample_stride + (int64_t)t * m.time_stride + idx];
}

template <class T>
struct PackArgs {
  LqgkSpec act, dyn;
  LqgkMat sigma0;
  int x, b, u, y;
  int nT;          // number of time steps (for the Qf default)
  int has_dyn;     // 0: gains-only call (dynamics-side constants are zero-filled)
};

// out(e) addresses element e of this sample's constant block.
template <class T, class Out>
LQGK_HD void pack_sample(const PackArgs<T>& a, int s, int t, Out&& out) {
  const CLayout cl(a.x, a.b, a.u, a.y);
  const int x = a.x, b = a.b, u = a.u, y = a.y;
  auto A_a = [&](int i, int j) { return mat_at<T>(a.act.A, s, t, i * b + j); };
  auto B_a = [&](int i, int j) { return mat_at<T>(a.act.B, s, t, i * u + j); };
  auto F_a = [&](int i, int j) { return mat_at<T>(a.act.F, s, t, i * b + j); };
  auto V_a = [&](int i, int j) { return mat_at<T>(a.act.V, s, t, i * b + j); };
  auto W_a = [&](int i, int j) { return mat_at<T>(a.act.W, s, t, i * y + j); };
  for (int i = 0; i < b; ++i)
    for (int j = 0; j < b; ++j) out(cl.Aa + i * b + j) = A_a(i, j);
  for (int i = 0; i < b * u; ++i) out(cl.Ba + i) = mat_at<T>(a.act.B, s, t, i);
  for (int i = 0; i < y * b; ++i) out(cl.Fa + i) = a.act.F.ptr ? mat_at<T>(a.act.F, s, t, i) : 0.0;
  for (int i = 0; i < b; ++i)
    for (int j = 0; j <= i; ++j) {
      out(cl.Q + sidx(i, j)) = a.act.Q.ptr ? 0.5 * (mat_at<T>(a.act.Q, s, t, i * b + j) + mat_at<T>(a.act.Q, s, t, j * b + i)) : 0.0;
      double qf;
      if (a.act.Qf.ptr) qf = 0.5 * (mat_at<T>(a.act.Qf, s, 0, i * b + j) + mat_at<T>(a.act.Qf, s, 0, j * b + i));
      else qf = a.act.Q.ptr ? 0.5 * (mat_at<T>(a.act.Q, s, a.nT - 1, i * b + j) + mat_at<T>(a.act.Q, s, a.nT - 1, j * b + i)) : 0.0;
      out(cl.Qf + sidx(i, j)) = qf;
      double vv = 0.0, v0 = 0.0;
      if (a.act.V.ptr)
        for (int k = 0; k < b; ++k) {
          vv += V_a(i, k) * V_a(j, k);
          v0 += mat_at<T>(a.act.V, s, 0, i * b + k) * mat_at<T>(a.act.V, s, 0, j * b + k);
        }
      out(cl.VVa + sidx(i, j)) = vv;
      out(cl.Sig0 + sidx(i, j)) = a.sigma0.ptr ? 0.5 * (mat_at<T>(a.sigma0, s, 0, i * b + j) + mat_at<T>(a.sigma0, s, 0, j * b + i)) : v0;
    }
  for (int i = 0; i < u; ++i)
    for (int j = 0; j <= i; ++j)
      out(cl.R + sidx(i, j)) = a.act.R.ptr ? 0.5 * (mat_at<T>(a.act.R, s, t, i * u + j) + mat_at<T>(a.act.R, s, t, j * u + i)) : 0.0;
  for (int i = 0; i < y; ++i)
    for (int j = 0; j <= i; ++j) {
      double ww = 0.0;
      if (a.act.W.ptr)
        for (int k = 0; k < y; ++k) ww += W_a(i, k) * W_a(j, k);
      out(cl.WWa + sidx(i, j)) = ww;
    }
  // affine terms (gains API)
  for (int i = 0; i < b; ++i) out(cl.q + i) = a.act.q.ptr ? mat_at<T>(a.act.q, s, t, i) : 0.0;
  for (int i = 0; i < u; ++i) out(cl.r + i) = a.act.r.ptr ? mat_at<T>(a.act.r, s, t, i) : 0.0;
  for (int i = 0; i < u * b; ++i) out(cl.P + i) = a.act.P.ptr ? mat_at<T>(a.act.P, s, t, i) : 0.0;
  for (int i = 0; i < b; ++i) out(cl.qf + i) = a.act.qf.ptr ? mat_at<T>(a.act.qf, s, 0, i) : 0.0;
  if (!a.has_dyn) {
    for (int e = cl.Ad; e < cl.q; ++e) out(e) = 0.0;
    return;
  }
  auto A_d = [&](int i, int j) { return mat_at<T>(a.dyn.A, s, t, i * x + j); };
  auto B_d = [&](int i, int j) { return mat_at<T>(a.dyn.B, s, t, i * u + j); };
  auto F_d = [&](int i, int j) { return mat_at<T>(a.dyn.F, s, t, i * x + j); };
  auto V_d = [&](int i, int j) { return mat_at<T>(a.dyn.V, s, t, i * x + j); };
  auto W_d = [&](int i, int j) { return mat_at<T>(a.dyn.W, s, t, i * y + j); };
  for (int i = 0; i < x * x; ++i) out(cl.Ad + i) = mat_at<T>(a.dyn.A, s, t, i);
  for (int i = 0; i < x * u; ++i) out(cl.Bd + i) = mat_at<T>(a.dyn.B, s, t, i);
  for (int k = 0; k < y; ++k) {
    for (int j = 0; j < x; ++j) {                       // FAd = Fd Ad
      double v = 0.0;
      for (int i = 0; i < x; ++i) v += F_d(k, i) * A_d(i, j);
      out(cl.FAd + k * x + j) = v;
    }
    for (int j = 0; j < b; ++j) {                       // FAa = Fa Aa
      double v = 0.0;
      for (int i = 0; i < b; ++i) v += F_a(k, i) * A_a(i, j);
      out(cl.FAa + k * b + j) = v;
    }
    for (int m = 0; m < u; ++m) {                       // D = Fd Bd - Fa Ba
      double v = 0.0;
      for (int i = 0; i < x; ++i) v += F_d(k, i) * B_d(i, m);
      for (int i = 0; i < b; ++i) v -= F_a(k, i) * B_a(i, m);
      out(cl.Dm + k * u + m) = v;
    }
  }
  for (int i = 0; i < x; ++i)
    for (int j = 0; j <= i; ++j) {                      // N11 = Vd Vd^T
      double v = 0.0;
      for (int k = 0; k < x; ++k) v += V_d(i, k) * V_d(j, k);
      out(cl.N11 + sidx(i, j)) = v;
    }
  for (int k = 0; k < y; ++k)
    for (int j = 0; j < x; ++j) {                       // FN = Fd N11
      double v = 0.0;
      for (int i = 0; i < x; ++i) v += F_d(k, i) * (double)out(cl.N11 + sidx(i, j));
      out(cl.FN + k * x + j) = v;
    }
  for (int k = 0; k < y; ++k)
    for (int m = 0; m <= k; ++m) {                      // Om = FN Fd^T + Wd Wd^T
      double v = 0.0;
      for (int j = 0; j < x; ++j) v += (double)out(cl.FN + k * x + j) * F_d(m, j);
      for (int j = 0; j < y; ++j) v += W_d(k, j) * W_d(m, j);
      out(cl.Om + sidx(k, m)) = v;
    }
}

template <class T>
struct UnpackArgs {
  LqgkSpec act, dyn;       // base matrices (time step 0)
  LqgkMat sigma0;
  LqgkSpecGrad gact, gdyn;
  LqgkMatGrad gsigma0;
  int x, b, u, y;
};

constexpr int LQGK_MAXDIM = 16;

template <class T>
LQGK_HD void store_grad(const LqgkMatGrad& g, int s, int idx, double v) {
  ((T*)g.ptr)[(int64_t)s * g.sample_stride + idx] = (T)v;
}

// acc(e): accumulated cotangent of derived constant e; cst(e): the derived constants themselves.  DYN = false: a call
// without a dynamics spec (the gains adjoint), whose a.dyn is empty: the actor's gradients only.
template <class T, bool DYN = true, class Acc, class Cst>
LQGK_HD void unpack_sample(const UnpackArgs<T>& a, int s, Acc&& acc, Cst&& cst) {
  const CLayout cl(a.x, a.b, a.u, a.y);
  const int x = a.x, b = a.b, u = a.u, y = a.y;
  auto A_a = [&](int i, int j) { return mat_at<T>(a.act.A, s, 0, i * b + j); };
  auto B_a = [&](int i, int j) { return mat_at<T>(a.act.B, s, 0, i * u + j); };
  auto F_a = [&](int i, int j) { return mat_at<T>(a.act.F, s, 0, i * b + j); };
  auto A_d = [&](int i, int j) { return mat_at<T>(a.dyn.A, s, 0, i * x + j); };
  auto B_d = [&](int i, int j) { return mat_at<T>(a.dyn.B, s, 0, i * u + j); };
  auto F_d = [&](int i, int j) { return mat_at<T>(a.dyn.F, s, 0, i * x + j); };
  // ---- actor
  if (a.gact.A.ptr)
    for (int i = 0; i < b; ++i)
      for (int j = 0; j < b; ++j) {                       // A_a: acc.Aa + Fa^T acc.FAa
        double v = acc(cl.Aa + i * b + j);
        for (int k = 0; k < y; ++k) v += F_a(k, i) * acc(cl.FAa + k * b + j);
        store_grad<T>(a.gact.A, s, i * b + j, v);
      }
  if (a.gact.B.ptr)
    for (int i = 0; i < b; ++i)
      for (int m = 0; m < u; ++m) {                       // B_a: acc.Ba - Fa^T acc.D
        double v = acc(cl.Ba + i * u + m);
        for (int k = 0; k < y; ++k) v -= F_a(k, i) * acc(cl.Dm + k * u + m);
        store_grad<T>(a.gact.B, s, i * u + m, v);
      }
  if (a.gact.F.ptr)
    for (int k = 0; k < y; ++k)
      for (int j = 0; j < b; ++j) {                       // F_a: acc.Fa + acc.FAa Aa^T - acc.D Ba^T
        double v = acc(cl.Fa + k * b + j);
        for (int i = 0; i < b; ++i) v += acc(cl.FAa + k * b + i) * A_a(j, i);
        for (int m = 0; m < u; ++m) v -= acc(cl.Dm + k * u + m) * B_a(j, m);
        store_grad<T>(a.gact.F, s, k * b + j, v);
      }
  if (a.gact.V.ptr)
    for (int i = 0; i < b; ++i)
      for (int j = 0; j < b; ++j) {                       // V_a: 2 (acc.VVa [+ acc.Sig0]) V
        double v = 0.0;
        for (int k = 0; k < b; ++k) {
          double g = acc(cl.VVa + sidx(i, k));
          if (!a.sigma0.ptr) g += acc(cl.Sig0 + sidx(i, k));
          v += 2.0 * g * mat_at<T>(a.act.V, s, 0, k * b + j);
        }
        store_grad<T>(a.gact.V, s, i * b + j, v);
      }
  if (a.gact.W.ptr)
    for (int i = 0; i < y; ++i)
      for (int j = 0; j < y; ++j) {
        double v = 0.0;
        for (int k = 0; k < y; ++k) v += 2.0 * acc(cl.WWa + sidx(i, k)) * mat_at<T>(a.act.W, s, 0, k * y + j);
        store_grad<T>(a.gact.W, s, i * y + j, v);
      }
  if (a.gact.Q.ptr)
    for (int i = 0; i < b; ++i)
      for (int j = 0; j < b; ++j) {
        double v = acc(cl.Q + sidx(i, j));
        if (!a.act.Qf.ptr) v += acc(cl.Qf + sidx(i, j));
        store_grad<T>(a.gact.Q, s, i * b + j, v);
      }
  if (a.gact.Qf.ptr)
    for (int i = 0; i < b; ++i)
      for (int j = 0; j < b; ++j) store_grad<T>(a.gact.Qf, s, i * b + j, a.act.Qf.ptr ? acc(cl.Qf + sidx(i, j)) : 0.0);
  if (a.gact.R.ptr)
    for (int i = 0; i < u; ++i)
      for (int j = 0; j < u; ++j) store_grad<T>(a.gact.R, s, i * u + j, acc(cl.R + sidx(i, j)));
  if (a.gsigma0.ptr)
    for (int i = 0; i < b; ++i)
      for (int j = 0; j < b; ++j) store_grad<T>(a.gsigma0, s, i * b + j, a.sigma0.ptr ? acc(cl.Sig0 + sidx(i, j)) : 0.0);
  if constexpr (!DYN) return;
  // ---- dynamics
  if (a.gdyn.A.ptr)
    for (int i = 0; i < x; ++i)
      for (int j = 0; j < x; ++j) {                       // A_d: acc.Ad + Fd^T acc.FAd
        double v = acc(cl.Ad + i * x + j);
        for (int k = 0; k < y; ++k) v += F_d(k, i) * acc(cl.FAd + k * x + j);
        store_grad<T>(a.gdyn.A, s, i * x + j, v);
      }
  if (a.gdyn.B.ptr)
    for (int i = 0; i < x; ++i)
      for (int m = 0; m < u; ++m) {                       // B_d: acc.Bd + Fd^T acc.D
        double v = acc(cl.Bd + i * u + m);
        for (int k = 0; k < y; ++k) v += F_d(k, i) * acc(cl.Dm + k * u + m);
        store_grad<T>(a.gdyn.B, s, i * u + m, v);
      }
  // FNb = acc.FN + Omb Fd  (y x x)
  double FNb[LQGK_MAXDIM * LQGK_MAXDIM];
  for (int k = 0; k < y; ++k)
    for (int j = 0; j < x; ++j) {
      double v = acc(cl.FN + k * x + j);
      for (int m = 0; m < y; ++m) v += acc(cl.Om + sidx(k, m)) * F_d(m, j);
      FNb[k * x + j] = v;
    }
  if (a.gdyn.F.ptr)
    for (int k = 0; k < y; ++k)
      for (int j = 0; j < x; ++j) {                       // F_d: acc.FAd Ad^T + acc.D Bd^T + Omb FN + FNb N11
        double v = 0.0;
        for (int i = 0; i < x; ++i) v += acc(cl.FAd + k * x + i) * A_d(j, i);
        for (int m = 0; m < u; ++m) v += acc(cl.Dm + k * u + m) * B_d(j, m);
        for (int m = 0; m < y; ++m) v += acc(cl.Om + sidx(k, m)) * cst(cl.FN + m * x + j);
        for (int i = 0; i < x; ++i) v += FNb[k * x + i] * cst(cl.N11 + sidx(i, j));
        store_grad<T>(a.gdyn.F, s, k * x + j, v);
      }
  if (a.gdyn.W.ptr)
    for (int i = 0; i < y; ++i)
      for (int j = 0; j < y; ++j) {
        double v = 0.0;
        for (int k = 0; k < y; ++k) v += 2.0 * acc(cl.Om + sidx(i, k)) * mat_at<T>(a.dyn.W, s, 0, k * y + j);
        store_grad<T>(a.gdyn.W, s, i * y + j, v);
      }
  if (a.gdyn.V.ptr) {
    double N11b[LQGK_MAXDIM * LQGK_MAXDIM];               // sym(acc.N11 + Fd^T FNb)
    for (int i = 0; i < x; ++i)
      for (int j = 0; j < x; ++j) {
        double v = 0.0;
        for (int k = 0; k < y; ++k) v += F_d(k, i) * FNb[k * x + j];
        N11b[i * x + j] = v;
      }
    for (int i = 0; i < x; ++i)
      for (int j = 0; j < x; ++j) {
        double v = 0.0;
        for (int k = 0; k < x; ++k)
          v += 2.0 * (acc(cl.N11 + sidx(i, k)) + 0.5 * (N11b[i * x + k] + N11b[k * x + i])) * mat_at<T>(a.dyn.V, s, 0, k * x + j);
        store_grad<T>(a.gdyn.V, s, i * x + j, v);
      }
  }
}

}  // namespace lqgk
