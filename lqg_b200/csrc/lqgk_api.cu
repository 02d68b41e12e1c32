// lqgk_api.cu -- extern "C" entry points of liblqgk.so (see include/lqgk.h): validation, dimension dispatch,
// workspace planning, chunking over parameter samples and the kernel launch sequence.
#include <cuda_runtime.h>
#include <curand_kernel.h>

#include <algorithm>
#include <cstdio>

#include "../../include/lqgk.h"
#include "lqgk_run.cuh"

using namespace lqgk;

namespace lqgk {
thread_local int g_launches = 0;
thread_local Profiler g_prof;
thread_local int g_streams = 1;
thread_local int g_contrib_warps = 0;    // 0 = 30 warps per SM of the current device
thread_local DeviceInfo g_dev;
thread_local int g_aux_streams = 6;
thread_local int g_warp_cov_max_samples = 512;   // measured crossover between 512 and 1,024 samples (profiles/r01_e_*.md)
thread_local StreamPool g_pool;
thread_local int g_pipe_max_samples = 1 << 30;   // measured: 1.2-1.4x at 8..8,192 samples, +2 % at 65,536 (profiles/r02_g_pipeline.md)
thread_local int g_pipe_segments = 6;
}

namespace {

// (the workspace and stream come last, as in every entry point's parameters)
template <class T>
int dispatch(Call& c, void* ws, size_t ws_bytes, void* stream) {
  g_launches = 0;
  c.ws = ws; c.ws_bytes = ws_bytes; c.stream = (cudaStream_t)stream;
  if (int rc = validate(c)) return rc;
  return visit_tuple<Tuples::compiled>(call_key(*c.dims, c.mode), LQGK_E_UNSUPPORTED, [&](auto dm, auto) {
    using R = Runner<decltype(dm)>;
    return std::is_same<T, float>::value ? R::run_f32(c) : R::run_f64(c);
  });
}

size_t workspace_bytes(const LqgkDims& d, int mode, int32_t max_chunk) {
  return visit_tuple<Tuples::compiled>(call_key(d, mode), (size_t)0,
                                       [&](auto dm, auto) { return Runner<decltype(dm)>::plan_bytes(d, mode, max_chunk); });
}

template <class T>
int pack_obs(int32_t N, int32_t T1, int32_t d, const T* x, float* x_tm, void* stream) {
  g_launches = 0;
  if (int rc = check_pack_obs(N, T1, d, x, x_tm)) return rc;
  size_t total = (size_t)N * T1 * d;
  k_pack_obs<T><<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(N, T1, d, x, x_tm);
  LQGK_LAUNCH_CHECK();
  return LQGK_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------- batched simulator
// System.simulate (lqg/system.py:62-140) for S parameter samples x N trials: one thread per trial runs the closed loop
//   u = L_t xhat + l_t;  x <- A_d x + B_d u + V_d eps_t;  y = F_d x + W_d eta_t;  xp = A_a xhat + B_a u;  xhat <- xp + K_t (y - F_a xp)
// in FP64 with standard-normal draws from a Philox4x32-10 counter stream (subsequence = trial index; the reference's JAX
// threefry stream cannot be reproduced, so the samples differ and the distribution does not).  Generic in the dimensions
// (run-time x, b, u, y <= SIM_MAX): it is a data generator, not a hot path.
constexpr int SIM_MAX = 40;
template <class T>
struct SimArgs {
  LqgkSpec act, dyn;
  const T *L, *l, *K, *x0, *xhat0;
  T *x_out, *xhat_out, *y_out, *u_out;
  int S, N, Tn, x, b, u, y;
  unsigned long long seed;
  // signal-dependent noise (extension, oracle/sdn_np.py: sdn_simulate): x += sum_i eps'_i C_i u,  y += sum_j eta'_j D_j x_new
  LqgkMat Cn, Dn;   // C[nc][x][u], D[nd][y][x] per sample (sample_stride 0 = shared)
  int nc, nd;
};
template <class T>
__global__ void k_simulate(SimArgs<T> a) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)a.S * a.N) return;
  const int s = (int)(idx / a.N);
  const int x = a.x, b = a.b, u = a.u, y = a.y, Tn = a.Tn;
  curandStatePhilox4_32_10_t rng;
  curand_init(a.seed, idx, 0, &rng);
  double xv[SIM_MAX], xh[SIM_MAX], xn[SIM_MAX], xp[SIM_MAX], yv[SIM_MAX], uv[SIM_MAX], nz[2 * SIM_MAX + 2 * SDN_MAX_TERMS + 4];
  for (int i = 0; i < x; ++i) xv[i] = a.x0 ? (double)a.x0[i] : 0.0;
  for (int i = 0; i < b; ++i) xh[i] = a.xhat0 ? (double)a.xhat0[i] : 0.0;
  T* xo = a.x_out + idx * (size_t)(Tn + 1) * x;
  T* ho = a.xhat_out ? a.xhat_out + idx * (size_t)(Tn + 1) * b : nullptr;
  T* yo = a.y_out ? a.y_out + idx * (size_t)Tn * y : nullptr;
  T* uo = a.u_out ? a.u_out + idx * (size_t)Tn * u : nullptr;
  for (int i = 0; i < x; ++i) xo[i] = (T)xv[i];
  if (ho) for (int i = 0; i < b; ++i) ho[i] = (T)xh[i];
  for (int t = 0; t < Tn; ++t) {
    for (int k = 0; k < x + y + a.nc + a.nd; k += 4) {   // (nc = nd = 0: the same stream as without the extension)
      float4 g = curand_normal4(&rng);
      nz[k] = g.x; nz[k + 1] = g.y; nz[k + 2] = g.z; nz[k + 3] = g.w;
    }
    const T* Lt = a.L + ((size_t)s * Tn + t) * u * b;
    const T* Kt = a.K + ((size_t)s * Tn + t) * b * y;
    for (int i = 0; i < u; ++i) {                                   // u = L xhat + l
      double v = a.l ? (double)a.l[((size_t)s * Tn + t) * u + i] : 0.0;
      for (int j = 0; j < b; ++j) v += (double)Lt[i * b + j] * xh[j];
      uv[i] = v;
    }
    for (int i = 0; i < x; ++i) {                                   // x <- A x + B u + V eps
      double v = 0.0;
      for (int j = 0; j < x; ++j) v += mat_at<T>(a.dyn.A, s, t, i * x + j) * xv[j] + mat_at<T>(a.dyn.V, s, t, i * x + j) * nz[j];
      for (int j = 0; j < u; ++j) v += mat_at<T>(a.dyn.B, s, t, i * u + j) * uv[j];
      xn[i] = v;
    }
    for (int q = 0; q < a.nc; ++q)                                  // control-dependent noise: + eps'_q C_q u
      for (int i = 0; i < x; ++i) {
        double v = 0.0;
        for (int j = 0; j < u; ++j) v += mat_at<T>(a.Cn, s, 0, (q * x + i) * u + j) * uv[j];
        xn[i] += nz[x + y + q] * v;
      }
    for (int i = 0; i < x; ++i) xv[i] = xn[i];
    for (int i = 0; i < y; ++i) {                                   // y = F x + W eta
      double v = 0.0;
      for (int j = 0; j < x; ++j) v += mat_at<T>(a.dyn.F, s, t, i * x + j) * xv[j];
      for (int j = 0; j < y; ++j) v += mat_at<T>(a.dyn.W, s, t, i * y + j) * nz[x + j];
      yv[i] = v;
    }
    for (int q = 0; q < a.nd; ++q)                                  // state-dependent observation noise: + eta'_q D_q x
      for (int i = 0; i < y; ++i) {
        double v = 0.0;
        for (int j = 0; j < x; ++j) v += mat_at<T>(a.Dn, s, 0, (q * y + i) * x + j) * xv[j];
        yv[i] += nz[x + y + a.nc + q] * v;
      }
    for (int i = 0; i < b; ++i) {                                   // xp = A_a xhat + B_a u
      double v = 0.0;
      for (int j = 0; j < b; ++j) v += mat_at<T>(a.act.A, s, t, i * b + j) * xh[j];
      for (int j = 0; j < u; ++j) v += mat_at<T>(a.act.B, s, t, i * u + j) * uv[j];
      xp[i] = v;
    }
    for (int i = 0; i < y; ++i) {                                   // innovation y - F_a xp (in place)
      double v = yv[i];
      for (int j = 0; j < b; ++j) v -= mat_at<T>(a.act.F, s, t, i * b + j) * xp[j];
      nz[i] = v;
    }
    for (int i = 0; i < b; ++i) {                                   // xhat <- xp + K innovation
      double v = xp[i];
      for (int j = 0; j < y; ++j) v += (double)Kt[i * y + j] * nz[j];
      xh[i] = v;
    }
    for (int i = 0; i < x; ++i) xo[(size_t)(t + 1) * x + i] = (T)xv[i];
    if (ho) for (int i = 0; i < b; ++i) ho[(size_t)(t + 1) * b + i] = (T)xh[i];
    if (yo) for (int i = 0; i < y; ++i) yo[(size_t)t * y + i] = (T)yv[i];
    if (uo) for (int i = 0; i < u; ++i) uo[(size_t)t * u + i] = (T)uv[i];
  }
}
namespace {
template <class T>
int simulate(const LqgkDims* d, const LqgkSpec* act, const LqgkSpec* dyn, const T* L, const T* l, const T* K, const T* x0, const T* xhat0,
             uint64_t seed, T* x_out, T* xhat_out, T* y_out, T* u_out, void* stream, const LqgkSdnNoise* nz = nullptr) {
  g_launches = 0;
  if (!d || !act || !dyn || !L || !K || !x_out) return LQGK_E_INVALID;
  if (d->S <= 0 || d->N <= 0 || d->T <= 0 || d->x <= 0 || d->b <= 0 || d->u <= 0 || d->y <= 0) return LQGK_E_INVALID;
  if (d->x > SIM_MAX || d->b > SIM_MAX || d->u > SIM_MAX || d->y > SIM_MAX) return LQGK_E_UNSUPPORTED;
  if (need_closed_loop(*act, *dyn, false) || check_noise(nz)) return LQGK_E_INVALID;
  SimArgs<T> a{*act, *dyn, L, l, K, x0, xhat0, x_out, xhat_out, y_out, u_out, d->S, d->N, d->T, d->x, d->b, d->u, d->y, seed};
  a.Cn = LqgkMat{nullptr, 0, 0}; a.Dn = LqgkMat{nullptr, 0, 0}; a.nc = 0; a.nd = 0;
  if (nz) { a.Cn = nz->C; a.Dn = nz->D; a.nc = nz->nc; a.nd = nz->nd; }
  const size_t total = (size_t)d->S * d->N;
  k_simulate<T><<<(unsigned)((total + 63) / 64), 64, 0, (cudaStream_t)stream>>>(a);
  LQGK_LAUNCH_CHECK();
  return LQGK_OK;
}

int sdn_loglik(const LqgkDims* d, const LqgkSpec* act, const LqgkSpec* dyn, const LqgkSdnNoise* nz, const void* L, const void* K,
               const float* x_tm, void* ll_out, bool f64, void* stream) {
  g_launches = 0;
  SdnLikArgs a;
  if (int rc = sdn_lik_args(d, act, dyn, nz, L, K, x_tm, ll_out, a)) return rc;
  // the tuples of the main path launch from their own objects (lqgk_inst.cu), the FP64-only ones from this one
  return visit_tuple<Tuples::small_and_fp64_only>(full_key(*d), LQGK_E_UNSUPPORTED, [&](auto dm, auto fp64_only) {
    using DM = decltype(dm);
    if constexpr (decltype(fp64_only)::value) return launch_sdn_loglik<DM>(a, f64, (cudaStream_t)stream);
    else return Runner<DM>::run_sdn_loglik(a, f64, (cudaStream_t)stream);
  });
}
int sdn_gains(const LqgkSdnDims* d, const LqgkSdnSpec* sp, double* L_out, double* K_out, double* cost_out, void* stream, int filter_form) {
  g_launches = 0;
  SdnArgs a;
  if (int rc = sdn_gains_args(d, sp, L_out, K_out, cost_out, filter_form, a)) return rc;
  return visit_tuple<Tuples::small>(TupleKey{ANY, d->b, d->u, d->y, ANY}, LQGK_E_UNSUPPORTED,
                                    [&](auto dm, auto) { return Runner<decltype(dm)>::run_sdn(a, (cudaStream_t)stream); });
}
}  // namespace

// FMA-saturating micro-kernels: the measured FP32 / FP64 CUDA-core peaks used as roofline denominators.
template <class T>
__global__ void k_peak_fma(int iters, T* sink) {
  T a[8];
  for (int i = 0; i < 8; ++i) a[i] = (T)(threadIdx.x + i) * (T)1e-3;
  const T m = (T)0.999, c = (T)1e-4;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = a[i] * m + c;
    }
  }
  T s = 0;
  for (int i = 0; i < 8; ++i) s += a[i];
  if (s == (T)123456.789) sink[0] = s;
}
extern "C" {

int lqgk_sdn_gains_f64(const LqgkSdnDims* d, const LqgkSdnSpec* sp, double* L_out, double* K_out, double* cost_out, void* stream) {
  return sdn_gains(d, sp, L_out, K_out, cost_out, stream, 0);
}
int lqgk_sdn_gains_filter_f64(const LqgkSdnDims* d, const LqgkSdnSpec* sp, double* L_out, double* K_out, double* cost_out, void* stream) {
  return sdn_gains(d, sp, L_out, K_out, cost_out, stream, 1);
}

int lqgk_sdn_loglik_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkSdnNoise* noise, const float* L,
                        const float* K, const float* x_tm, float* ll_out, void* stream) {
  return sdn_loglik(dims, actor, dynamics, noise, L, K, x_tm, ll_out, false, stream);
}
int lqgk_sdn_loglik_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkSdnNoise* noise, const double* L,
                        const double* K, const float* x_tm, double* ll_out, void* stream) {
  return sdn_loglik(dims, actor, dynamics, noise, L, K, x_tm, ll_out, true, stream);
}

int lqgk_lqr_backward_f32(const LqgkDims* dims, const LqgkSpec* actor, double eps, float* L_out, float* l_out, float* H_out,
                          void* ws, size_t ws_bytes, void* stream) {
  Call c;
  c.mode = LQGK_MODE_GAINS; c.dims = dims; c.act = actor; c.eps = eps; c.L_out = L_out; c.l_out = l_out; c.H_out = H_out;
  return dispatch<float>(c, ws, ws_bytes, stream);
}
int lqgk_lqr_backward_f64(const LqgkDims* dims, const LqgkSpec* actor, double eps, double* L_out, double* l_out, double* H_out,
                          void* ws, size_t ws_bytes, void* stream) {
  Call c;
  c.mode = LQGK_MODE_GAINS; c.dims = dims; c.act = actor; c.eps = eps; c.L_out = L_out; c.l_out = l_out; c.H_out = H_out;
  return dispatch<double>(c, ws, ws_bytes, stream);
}
int lqgk_kf_forward_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, float* K_out, void* ws,
                        size_t ws_bytes, void* stream) {
  Call c;
  c.mode = LQGK_MODE_GAINS; c.dims = dims; c.act = actor; c.sigma0 = sigma0; c.K_out = K_out;
  return dispatch<float>(c, ws, ws_bytes, stream);
}
int lqgk_kf_forward_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, double* K_out, void* ws,
                        size_t ws_bytes, void* stream) {
  Call c;
  c.mode = LQGK_MODE_GAINS; c.dims = dims; c.act = actor; c.sigma0 = sigma0; c.K_out = K_out;
  return dispatch<double>(c, ws, ws_bytes, stream);
}
int lqgk_gains_vjp_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, double eps, const float* L_bar,
                       const float* K_bar, const LqgkSpecGrad* ga, const LqgkMatGrad* gs, void* ws, size_t ws_bytes, void* stream) {
  LqgkSpec base;
  Call c = gains_vjp_call(dims, actor, sigma0, eps, L_bar, K_bar, ga, gs, base);
  return dispatch<float>(c, ws, ws_bytes, stream);
}
int lqgk_gains_vjp_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, double eps, const double* L_bar,
                       const double* K_bar, const LqgkSpecGrad* ga, const LqgkMatGrad* gs, void* ws, size_t ws_bytes, void* stream) {
  LqgkSpec base;
  Call c = gains_vjp_call(dims, actor, sigma0, eps, L_bar, K_bar, ga, gs, base);
  return dispatch<double>(c, ws, ws_bytes, stream);
}
int lqgk_loglik_fwd_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0,
                        const float* x_tm, float* ll_out, void* ws, size_t ws_bytes, void* stream) {
  Call c;
  c.mode = LQGK_MODE_FWD; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.ll_out = ll_out;
  return dispatch<float>(c, ws, ws_bytes, stream);
}
int lqgk_loglik_fwd_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0,
                        const float* x_tm, double* ll_out, void* ws, size_t ws_bytes, void* stream) {
  Call c;
  c.mode = LQGK_MODE_FWD; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.ll_out = ll_out;
  return dispatch<double>(c, ws, ws_bytes, stream);
}
int lqgk_loglik_vjp_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0,
                        const float* x_tm, const float* ll_bar, float* ll_out, const LqgkSpecGrad* ga, const LqgkSpecGrad* gd,
                        const LqgkMatGrad* gs, void* ws, size_t ws_bytes, void* stream) {
  Call c;
  c.mode = LQGK_MODE_VJP; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.ll_bar = ll_bar;
  c.ll_out = ll_out; c.gact = ga; c.gdyn = gd; c.gsig0 = gs;
  return dispatch<float>(c, ws, ws_bytes, stream);
}
int lqgk_loglik_vjp_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0,
                        const float* x_tm, const double* ll_bar, double* ll_out, const LqgkSpecGrad* ga, const LqgkSpecGrad* gd,
                        const LqgkMatGrad* gs, void* ws, size_t ws_bytes, void* stream) {
  Call c;
  c.mode = LQGK_MODE_VJP; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.ll_bar = ll_bar;
  c.ll_out = ll_out; c.gact = ga; c.gdyn = gd; c.gsig0 = gs;
  return dispatch<double>(c, ws, ws_bytes, stream);
}

int lqgk_moments_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0, const float* x_tm,
                     float* mu_out, float* Sigma_out, void* ws, size_t ws_bytes, void* stream) {
  Call c;
  c.mode = LQGK_MODE_MOMENTS; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.mu_out = mu_out;
  c.Sig_out = Sigma_out;
  return dispatch<float>(c, ws, ws_bytes, stream);
}
int lqgk_moments_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0, const float* x_tm,
                     double* mu_out, double* Sigma_out, void* ws, size_t ws_bytes, void* stream) {
  Call c;
  c.mode = LQGK_MODE_MOMENTS; c.dims = dims; c.act = actor; c.dyn = dynamics; c.sigma0 = sigma0; c.x_tm = x_tm; c.mu_out = mu_out;
  c.Sig_out = Sigma_out;
  return dispatch<double>(c, ws, ws_bytes, stream);
}
int lqgk_simulate_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const float* L, const float* l, const float* K,
                      const float* x0, const float* xhat0, uint64_t seed, float* x_out, float* xhat_out, float* y_out, float* u_out,
                      void* stream) {
  return simulate<float>(dims, actor, dynamics, L, l, K, x0, xhat0, seed, x_out, xhat_out, y_out, u_out, stream);
}
int lqgk_simulate_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const double* L, const double* l, const double* K,
                      const double* x0, const double* xhat0, uint64_t seed, double* x_out, double* xhat_out, double* y_out, double* u_out,
                      void* stream) {
  return simulate<double>(dims, actor, dynamics, L, l, K, x0, xhat0, seed, x_out, xhat_out, y_out, u_out, stream);
}

int lqgk_sdn_simulate_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkSdnNoise* noise, const float* L,
                          const float* l, const float* K, const float* x0, const float* xhat0, uint64_t seed, float* x_out, float* xhat_out,
                          float* y_out, float* u_out, void* stream) {
  return simulate<float>(dims, actor, dynamics, L, l, K, x0, xhat0, seed, x_out, xhat_out, y_out, u_out, stream, noise);
}
int lqgk_sdn_simulate_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkSdnNoise* noise, const double* L,
                          const double* l, const double* K, const double* x0, const double* xhat0, uint64_t seed, double* x_out,
                          double* xhat_out, double* y_out, double* u_out, void* stream) {
  return simulate<double>(dims, actor, dynamics, L, l, K, x0, xhat0, seed, x_out, xhat_out, y_out, u_out, stream, noise);
}

int lqgk_pack_obs_f32(int32_t N, int32_t T1, int32_t d, const float* x, float* x_tm, void* stream) {
  return pack_obs<float>(N, T1, d, x, x_tm, stream);
}
int lqgk_pack_obs_f64(int32_t N, int32_t T1, int32_t d, const double* x, float* x_tm, void* stream) {
  return pack_obs<double>(N, T1, d, x, x_tm, stream);
}

size_t lqgk_workspace_bytes(const LqgkDims* dims, int mode, int32_t max_chunk) {
  return dims ? workspace_bytes(*dims, mode, max_chunk) : 0;
}

int lqgk_dims_supported(const LqgkDims* dims) {
  return dims && visit_tuple<Tuples::compiled>(full_key(*dims), 0, [](auto, auto) { return 1; });
}

const char* lqgk_strerror(int code) {
  switch (code) {
    case LQGK_OK: return "ok";
    case LQGK_E_INVALID: return "invalid argument (null pointer, non-positive dimension or misaligned buffer)";
    case LQGK_E_UNSUPPORTED: return "unsupported: dimension tuple not compiled in, or time-varying spec (or cross cost P) passed to an adjoint";
    case LQGK_E_WORKSPACE: return "workspace too small for one 32-sample chunk (see lqgk_workspace_bytes)";
    case LQGK_E_CUDA: return "CUDA runtime error";
    case LQGK_E_NOT_INITIALISED: return "internal streams missing while the caller's stream is being captured: call lqgk_init() on this thread and device before capturing";
    default: return "unknown error";
  }
}
int lqgk_init(int max_sample_slices) {
  // everything an entry point may need later on this thread and device, created now: the internal streams / events (sample
  // slices + 3 auxiliary streams per slice) and the cached SM count.  After this no entry point creates CUDA objects, so calls
  // may be captured into CUDA graphs (which is how XLA may run an FFI handler).
  if (max_sample_slices < 1 || max_sample_slices > 32) return LQGK_E_INVALID;
  sm_count();
  return g_pool.ensure(3 * max_sample_slices);
}
int lqgk_set_streams(int n) {
  if (n < 1 || n > 32) return LQGK_E_INVALID;
  g_streams = n;
  return LQGK_OK;
}
int lqgk_set_contrib_warps(int n) {
  if (n < 1) return LQGK_E_INVALID;
  g_contrib_warps = n;
  return LQGK_OK;
}
int lqgk_set_warp_cov_max_samples(int n) {
  if (n < 0) return LQGK_E_INVALID;
  g_warp_cov_max_samples = n;
  return LQGK_OK;
}
int lqgk_set_pipeline(int max_samples, int segments) {
  if (max_samples < 0 || segments < 1 || segments > 64) return LQGK_E_INVALID;
  g_pipe_max_samples = max_samples;
  g_pipe_segments = segments;
  return LQGK_OK;
}
int lqgk_set_kernel_overlap(int mask) {
  if (mask < 0 || mask > 7) return LQGK_E_INVALID;
  g_aux_streams = mask;
  return LQGK_OK;
}
int lqgk_profile_enable(int on) {
  g_prof.on = on != 0;
  g_prof.used = 0;
  return LQGK_OK;
}
int lqgk_profile_timeline(float* start_ms, float* end_ms, int32_t* kind, int max_entries) {
  // start/end of every recorded launch relative to the first recorded event (call before lqgk_profile_read)
  int n = 0;
  if (g_prof.used < 2) return 0;
  for (size_t i = 0; i + 1 < g_prof.used && n < max_entries; i += 2, ++n) {
    if (cudaEventSynchronize(g_prof.ev[i + 1]) != cudaSuccess) return LQGK_E_CUDA;
    cudaEventElapsedTime(&start_ms[n], g_prof.ev[0], g_prof.ev[i]);
    cudaEventElapsedTime(&end_ms[n], g_prof.ev[0], g_prof.ev[i + 1]);
    kind[n] = g_prof.kinds[i / 2];
  }
  return n;
}
int lqgk_profile_read(float* ms_by_kind, int32_t* launches_by_kind, int nkinds) {
  if (!ms_by_kind || nkinds <= 0) return LQGK_E_INVALID;
  for (int i = 0; i < nkinds; ++i) { ms_by_kind[i] = 0.f; if (launches_by_kind) launches_by_kind[i] = 0; }
  for (size_t i = 0; i + 1 < g_prof.used; i += 2) {
    if (cudaEventSynchronize(g_prof.ev[i + 1]) != cudaSuccess) return LQGK_E_CUDA;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g_prof.ev[i], g_prof.ev[i + 1]) != cudaSuccess) return LQGK_E_CUDA;
    int k = g_prof.kinds[i / 2];
    if (k < nkinds) { ms_by_kind[k] += ms; if (launches_by_kind) launches_by_kind[k] += 1; }
  }
  g_prof.used = 0;
  return PK_COUNT;
}

int lqgk_peak_fma(int fp64, int iters, void* sink, void* stream, double* flop_out) {
  if (!sink || iters <= 0) return LQGK_E_INVALID;
  const int blocks = sm_count() * 8, threads = 256;
  if (fp64) k_peak_fma<double><<<blocks, threads, 0, (cudaStream_t)stream>>>(iters, (double*)sink);
  else k_peak_fma<float><<<blocks, threads, 0, (cudaStream_t)stream>>>(iters, (float*)sink);
  if (cudaPeekAtLastError() != cudaSuccess) return LQGK_E_CUDA;
  if (flop_out) *flop_out = 2.0 * 64.0 * (double)iters * blocks * threads;
  return LQGK_OK;
}

const char* lqgk_version(void) { return "lqgk 0.2.0 (sm_100a)"; }
const char* lqgk_last_cuda_error(void) { return cudaGetErrorString(cudaPeekAtLastError()); }
int lqgk_last_launch_count(void) { return g_launches; }

}  // extern "C"
