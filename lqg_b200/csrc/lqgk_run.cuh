// lqgk_run.cuh -- workspace planning, chunking over parameter samples and the kernel launch sequence for one
// dimension tuple.  Instantiated once per tuple by lqgk_inst.cu (compiled in parallel), called from lqgk_api.cu.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <vector>

#include "../../include/lqgk.h"
#include "lqgk_kernels.cuh"
#include "lqgk_bigw.cuh"
#include "lqgk_entry.h"
#include "lqgk_sdn.cuh"

namespace lqgk {

extern thread_local int g_launches;

// Optional per-kernel timing (bench.py): CUDA events recorded on the launching stream around every launch.
enum ProfKind { PK_PACK = 0, PK_LQR_FWD, PK_KF_FWD, PK_COV_FWD, PK_TRIAL_FWD, PK_MISC, PK_TRIAL_REV, PK_COV_REV, PK_KF_REV,
                PK_LQR_REV, PK_UNPACK, PK_COV_CONTRIB, PK_REDUCE, PK_COUNT };
struct Profiler {
  bool on = false;
  std::vector<cudaEvent_t> ev;   // pairs (start, stop)
  std::vector<int> kinds;
  size_t used = 0;
};
extern thread_local Profiler g_prof;

// Concurrent sample slices: the per-sample kernels are latency-bound (about one warp per scheduler), so a call splits
// its samples into up to g_streams slices that run the whole kernel sequence concurrently on internal non-blocking
// streams (forked from / joined to the caller's stream with events); each slice owns a part of the workspace.
extern thread_local int g_streams;
extern thread_local int g_contrib_warps;   // target number of (sample-group x time-range) warps of the contraction kernels
extern thread_local int g_aux_streams;   // 0: no internal auxiliary streams (no pipelined launch sequence); else allowed
// SM count of the calling thread's current device (queried once per device, never hard-coded): sizes the grids of the
// time-parallel kernels.
struct DeviceInfo {
  int device = -1, sms = 0;
};
extern thread_local DeviceInfo g_dev;
inline int sm_count() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != g_dev.device || g_dev.sms <= 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    g_dev.device = dev;
    g_dev.sms = n;
  }
  return g_dev.sms;
}

// Internal streams / events of the calling thread (one pool per thread and device).  lqgk_init() creates them up front;
// entry points only create what is missing when the caller's stream is NOT being captured into a CUDA graph (creating
// streams inside a capture is illegal) and otherwise return LQGK_E_NOT_INITIALISED.
struct StreamPool {
  static constexpr size_t NEV = 64;
  int device = -1;
  std::vector<cudaStream_t> streams;
  std::vector<cudaEvent_t> joins;
  cudaEvent_t fork = nullptr;
  std::vector<cudaEvent_t> evs;   // round-robin pool for intra-chunk dependencies (timing disabled)
  size_t ev_next = 0;
  cudaEvent_t next_event() { return evs[ev_next++ % evs.size()]; }
  bool ready(int n) const {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    return dev == device && fork && (int)streams.size() >= n && evs.size() >= NEV;
  }
  int ensure(int n) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return LQGK_E_CUDA;
    if (dev != device) {   // one pool per thread and device; streams of another device are simply abandoned
      streams.clear();
      joins.clear();
      evs.clear();
      fork = nullptr;
      device = dev;
    }
    if (!fork && cudaEventCreateWithFlags(&fork, cudaEventDisableTiming) != cudaSuccess) return LQGK_E_CUDA;
    while (evs.size() < NEV) {
      cudaEvent_t e;
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return LQGK_E_CUDA;
      evs.push_back(e);
    }
    while ((int)streams.size() < n) {
      cudaStream_t st;
      cudaEvent_t ev;
      // highest priority: the internal streams carry the latency-bound per-sample sweeps of the pipelined launch sequence, whose
      // small CTAs should get the first free SM resources when they compete with the (throughput-bound) per-trial kernels
      int prio_lo = 0, prio_hi = 0;
      cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
      if (cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, prio_hi) != cudaSuccess) return LQGK_E_CUDA;
      if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) return LQGK_E_CUDA;
      streams.push_back(st);
      joins.push_back(ev);
    }
    return LQGK_OK;
  }
  // what an entry point calls: never creates anything while `caller` is being captured
  int acquire(int n, cudaStream_t caller) {
    if (ready(n)) return LQGK_OK;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(caller, &cs) != cudaSuccess) return LQGK_E_CUDA;
    if (cs != cudaStreamCaptureStatusNone) return LQGK_E_NOT_INITIALISED;
    return ensure(n);
  }
};
extern thread_local StreamPool g_pool;
struct ProfScope {
  cudaStream_t st;
  bool active;
  ProfScope(int kind, cudaStream_t s) : st(s), active(g_prof.on) {
    if (!active) return;
    if (g_prof.used + 2 > g_prof.ev.size()) {
      cudaEvent_t a, b;
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      g_prof.ev.push_back(a);
      g_prof.ev.push_back(b);
    }
    g_prof.kinds.resize(g_prof.ev.size() / 2);
    g_prof.kinds[g_prof.used / 2] = kind;
    cudaEventRecord(g_prof.ev[g_prof.used], st);
  }
  ~ProfScope() {
    if (!active) return;
    cudaEventRecord(g_prof.ev[g_prof.used + 1], st);
    g_prof.used += 2;
  }
};

#define LQGK_LAUNCH_CHECK()                              \
  do {                                                   \
    ++g_launches;                                        \
    if (cudaPeekAtLastError() != cudaSuccess) return LQGK_E_CUDA; \
  } while (0)

constexpr size_t ALIGN = 256;
extern thread_local int g_warp_cov_max_samples;   // calls with at most this many samples use the warp-per-sample covariance kernels
// Pipelined launch sequence (VJP): chunks of at most g_pipe_max_samples samples cut every sequential sweep into
// g_pipe_segments time segments and run the sweeps of one direction as a software pipeline over internal streams.
extern thread_local int g_pipe_max_samples, g_pipe_segments;
inline size_t up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Large systems (joint dim > 12) take the warp-per-sample kernels of lqgk_bigw.cuh (see the kernel launchers below).
template <class DM>
constexpr bool is_big() { return DM::N > 12; }
// Workspace plan for one chunk of Sc (multiple of 32) samples.
struct Plan {
  size_t Sc = 0, bytes = 0;
  size_t cst = 0, acc = 0, L = 0, K = 0, l = 0, H = 0, Sric = 0, Pkf = 0, Cs = 0, Lbar = 0, Kbar = 0, rec = 0, ll = 0,
         sums = 0, hist = 0, w = 0, FU = 0, JS = 0, J0 = 0, SGB = 0, SGBI = 0, SFW = 0, KbarF = 0, scr = 0, xc = 0,
         carC = 0, carP = 0, carcb = 0;
};

template <class DM>
Plan make_plan(const LqgkDims& d, int mode, bool tv, size_t Sc) {
  Plan p;
  p.Sc = Sc;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = up(off + bytes, ALIGN); return o; };
  const size_t T = d.T, N = d.N;
  constexpr CLayout cl = DM::CL;
  p.cst = take(sizeof(double) * cl.total * Sc * (tv ? T : 1));
  p.L = take(sizeof(double) * T * DM::EL * Sc);
  p.K = take(sizeof(double) * T * DM::EK * Sc);
  if (mode == LQGK_MODE_GAINS) {
    p.l = take(sizeof(double) * T * DM::U * Sc);
    p.H = take(sizeof(double) * T * DM::U * DM::U * Sc);
  } else if (mode == LQGK_MODE_MOMENTS) {
    p.rec = take(sizeof(float) * Sc * T * DM::REC);
  } else if (mode == LQGK_MODE_GAINS_VJP) {
    p.acc = take(sizeof(double) * cl.total * Sc);
    p.Sric = take(sizeof(double) * T * DM::ES * Sc);
    p.Pkf = take(sizeof(double) * T * DM::EP * Sc);
    p.Lbar = take(sizeof(double) * T * DM::EL * Sc);
    p.Kbar = take(sizeof(double) * T * DM::EK * Sc);
    p.KbarF = take(sizeof(double) * T * DM::EK * Sc);
    p.carP = take(sizeof(double) * DM::B * DM::B * Sc);
  } else {
    p.rec = take(sizeof(float) * Sc * T * DM::REC);
    p.ll = take(sizeof(double) * Sc * N);
    const TrialGeom tg = trial_geom<DM>((int)N, (int)T);
    p.xc = take(sizeof(float) * (d.x_sample_stride != 0 ? Sc : 1) * (T + 1) * tg.NB * d.d * tg.ROW);   // repacked observations
  }
  if (mode == LQGK_MODE_VJP) {
    p.acc = take(sizeof(double) * cl.total * Sc);
    p.Sric = take(sizeof(double) * T * DM::ES * Sc);
    p.Pkf = take(sizeof(double) * T * DM::EP * Sc);
    p.Cs = take(sizeof(double) * T * DM::EC * Sc);
    p.Lbar = take(sizeof(double) * T * DM::EL * Sc);
    p.Kbar = take(sizeof(double) * T * DM::EK * Sc);
    p.KbarF = take(sizeof(double) * T * DM::EK * Sc);
    p.sums = take(sizeof(float) * Sc * T * DM::SUMP);
    {
      const TrialGeom tg = trial_geom<DM>((int)N, (int)T);
      p.hist = take(sizeof(float) * Sc * tg.nseg * tg.NB * DM::R * tg.ROW);   // checkpoints of the carried state
      // carries between the time segments of the pipelined launch sequence
      p.carcb = take(sizeof(float) * Sc * tg.NB * DM::R * tg.ROW);
      p.carC = take(sizeof(double) * DM::R * DM::R * Sc);
      p.carP = take(sizeof(double) * DM::B * DM::B * Sc);
    }
    p.w = take(sizeof(float) * Sc * N);
    using SR = CovSeqRev<DM>;
    p.FU = take(sizeof(lin_t) * T * SR::NSF * Sc);      // FP32 linearisation points (see lin_t)
    p.JS = take(sizeof(lin_t) * T * SR::NJS * Sc);
    p.J0 = take(sizeof(double) * DM::R * DM::D * Sc);
    p.SGB = take(sizeof(lin_t) * T * SR::NSGB * Sc);
    p.SGBI = take(sizeof(double) * SR::NSGB * Sc);
    p.SFW = take(sizeof(lin_t) * T * SR::NSF * Sc);
  }
  p.bytes = off;
  return p;
}

template <class DM>
size_t choose_chunk(const LqgkDims& d, int mode, bool tv, size_t ws_bytes, int32_t max_chunk) {
  size_t Spad = up((size_t)d.S, 32);
  size_t cap = Spad;
  if (max_chunk > 0) cap = std::min(cap, up((size_t)max_chunk, 32));
  if (ws_bytes == (size_t)-1) return cap;
  // plan size is (almost) linear in Sc: find the largest multiple of 32 that fits
  size_t lo = 0, hi = cap / 32;
  while (lo < hi) {
    size_t mid = (lo + hi + 1) / 2;
    if (make_plan<DM>(d, mode, tv, mid * 32).bytes <= ws_bytes) lo = mid; else hi = mid - 1;
  }
  return lo * 32;
}

template <class DM>
int set_smem(const void* fn, size_t bytes) {
  if (bytes > 48 * 1024) {
    if (bytes > 227 * 1024) return LQGK_E_UNSUPPORTED;
    if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) return LQGK_E_CUDA;
  }
  return LQGK_OK;
}

// ka, kb: range of checkpoint segments of this launch
template <class DM, int RT>
int launch_trial_fwd(cudaStream_t st, const float* rec, const float* xc, size_t xcs, int n, int N, int T, double* ll, float* hist,
                     int ka, int kb) {
  size_t smem = trial_smem_bytes<DM, RT, false>();
  int rc = set_smem<DM>((const void*)k_trial_fwd<DM, RT>, smem);
  if (rc) return rc;
  ProfScope ps_(PK_TRIAL_FWD, st);
  k_trial_fwd<DM, RT><<<(n + TRIAL_WARPS - 1) / TRIAL_WARPS, 32 * TRIAL_WARPS, smem, st>>>(rec, xc, xcs, n, N, T, ll, hist, ka, kb);
  LQGK_LAUNCH_CHECK();
  return LQGK_OK;
}
template <class DM, int RT>
int launch_trial_rev(cudaStream_t st, const float* rec, const float* xc, size_t xcs, const float* hist, const float* w, int n, int N, int T,
                     float* sums, float* cbcar, int ka, int kb) {
  size_t smem = trial_smem_bytes<DM, RT, true>();
  int rc = set_smem<DM>((const void*)k_trial_rev<DM, RT>, smem);
  if (rc) return rc;
  ProfScope ps_(PK_TRIAL_REV, st);
  k_trial_rev<DM, RT><<<(n + TRIAL_WARPS_REV - 1) / TRIAL_WARPS_REV, 32 * TRIAL_WARPS_REV, smem, st>>>(rec, xc, xcs, hist, w, n, N, T, sums, ka,
                                                                                                     kb, cbcar);
  LQGK_LAUNCH_CHECK();
  return LQGK_OK;
}

// ------------------------------------------------------------------------------------------------------- kernel launchers
// One launcher per stage of the likelihood path.  A launcher takes its stream and, for a sweep over time, the range of one
// pipeline segment ([t0, t1) in steps; [ka, kb) in checkpoint segments for the per-trial kernels).  It picks the kernel variant
// for the system size and the covariance mapping, sets the kernel's dynamic shared memory, times the launch (ProfScope) and
// checks it.
//
// Small systems (joint dim n <= 12) keep every matrix of a sample in registers (one thread per sample, fully unrolled
// templates) and its constants in shared memory, with sample-minor workspace arrays.  Few samples (a handful of conditions, a
// few hundred chains per GPU) leave the thread-per-sample covariance kernels with an idle GPU and every step costing one thread's
// instruction stream; calls with at most g_warp_cov_max_samples samples therefore run the large systems' warp-per-sample
// covariance kernels, which spread a step over 32 lanes (S = 8: covariance forward 3.3 -> 2.4 ms, sequential adjoint
// 2.5 -> 1.0 ms) and win up to ~1,000 samples.  The Riccati / Kalman sweeps stay thread-per-sample (3 x 3 products do not
// spread), hence GAINS_MINOR: the warp kernels read the sample-minor gains of those sweeps.
//
// Large systems (joint dim n > 12, e.g. the 24-dim delayed point-mass model of BASELINE config c4:
// TemporalDelayModel(PointMassBoundedActor, delay=2)): neither fits at n = 24 (576-entry joint matrices, ~900 derived
// constants per sample), and these systems come in thousands, not hundreds of thousands, of samples.  Their path therefore
// maps ONE WARP PER PARAMETER SAMPLE with the matrices in shared memory (lqgk_bigw.cuh: kw_lqr_fwd, kw_kf_fwd, kw_cov_fwd,
// kw_cov_seq_rev, kw_cov_contrib, kw_kf_rev, kw_lqr_rev) and sample-major workspace arrays.  The per-trial FP32 kernels
// (k_trial_fwd / k_trial_rev: warp per sample, lane = trial, TMA-staged records) are shared with the small-system path; only
// their ring geometry adapts to the record size.  The object is compiled with -DLQGK_BIG (rolled FP64 loops in the scalar
// helpers the lanes still call for the u x u / y x y / d x d factorisations).  kw_lqr_* and kw_kf_* take no time range: a
// large system always runs one segment.
template <class DM, class T>
struct Chunk {
  static constexpr bool BIG = is_big<DM>();
  static constexpr unsigned WTHR = 32 * BW_WARPS;   // threads per CTA of the warp-per-sample kernels
  const Call& c;
  const Plan& p;
  char* base;               // this slice's part of the workspace
  size_t s0;                // first sample of the chunk
  int n, npad, nblk, wblk;  // samples (valid, padded to 32); CTAs of the thread- and of the warp-per-sample kernels
  int Tn, N;
  bool tv;
  bool vjp;                 // the likelihood's adjoint: its buffers (covariance linearisation points, checkpoints, weights)
  bool keep;                // keep S_t and P_t for an adjoint (the likelihood's or the gains')
  bool warp_cov;            // covariance kernels one warp per sample (always for the large systems)
  size_t xcs = 0;           // element stride between the repacked observation sets in xc (repack_obs)

  double* D(size_t off) const { return (double*)(base + off); }
  float* F(size_t off) const { return (float*)(base + off); }
  size_t tstride() const { return tv ? (size_t)DM::CL.total * p.Sc : 0; }
  int rt() const { return trial_rt(N, trial_rt_max<DM>()); }

  int pack(cudaStream_t st) const {
    PackArgs<T> pa{};
    pa.act = *c.act;
    if (c.dyn) pa.dyn = *c.dyn;
    pa.sigma0 = c.sigma0 ? *c.sigma0 : LqgkMat{nullptr, 0, 0};
    pa.x = DM::X; pa.b = DM::B; pa.u = DM::U; pa.y = DM::Y; pa.nT = Tn; pa.has_dyn = c.dyn != nullptr;
    ProfScope ps_(PK_PACK, st);
    k_pack<T><<<dim3((npad + 127) / 128, tv ? Tn : 1), 128, 0, st>>>(pa, (int)s0, n, npad, D(p.cst), p.Sc, tstride(), tv ? Tn : 1);
    LQGK_LAUNCH_CHECK();
    return LQGK_OK;
  }
  // Riccati sweep, t down.  AFFINE (gains entry point): also l_t and H_t.  keep: keeps S_t for the adjoint.
  template <bool AFFINE>
  int lqr_fwd(cudaStream_t st) const {
    double *Sric = keep ? D(p.Sric) : nullptr, *l = AFFINE ? D(p.l) : nullptr, *H = AFFINE ? D(p.H) : nullptr;
    int rc;
    if constexpr (BIG) {
      const size_t smem = BigG<DM>::smem_lqr();
      if ((rc = set_smem<DM>((const void*)kw_lqr_fwd<DM, AFFINE>, smem))) return rc;
      ProfScope ps_(PK_LQR_FWD, st);
      kw_lqr_fwd<DM, AFFINE><<<wblk, WTHR, smem, st>>>(D(p.cst), p.Sc, npad, Tn, c.eps, D(p.L), keep, Sric, l, H);
      LQGK_LAUNCH_CHECK();
    } else {
      const size_t smem = sizeof(double) * 32 * (AFFINE ? LqrC<DM>::n_affine : LqrC<DM>::n);
      if ((rc = set_smem<DM>((const void*)k_lqr_fwd<DM, AFFINE>, smem))) return rc;
      ProfScope ps_(PK_LQR_FWD, st);
      k_lqr_fwd<DM, AFFINE><<<nblk, 32, smem, st>>>(D(p.cst), p.Sc, tstride(), Tn, c.eps, D(p.L), keep, Sric, l, H);
      LQGK_LAUNCH_CHECK();
    }
    return LQGK_OK;
  }
  // Kalman sweep, t up over [t0, t1).  keep: keeps P_t for the adjoint.
  int kf_fwd(cudaStream_t st, int t0, int t1) const {
    double* Pkf = keep ? D(p.Pkf) : nullptr;
    int rc;
    if constexpr (BIG) {
      const size_t smem = BigG<DM>::smem_kf();
      if ((rc = set_smem<DM>((const void*)kw_kf_fwd<DM>, smem))) return rc;
      ProfScope ps_(PK_KF_FWD, st);
      kw_kf_fwd<DM><<<wblk, WTHR, smem, st>>>(D(p.cst), p.Sc, npad, Tn, D(p.K), keep, Pkf);
      LQGK_LAUNCH_CHECK();
    } else {
      const size_t smem = sizeof(double) * 32 * KfC<DM>::n;
      if ((rc = set_smem<DM>((const void*)k_kf_fwd<DM>, smem))) return rc;
      ProfScope ps_(PK_KF_FWD, st);
      k_kf_fwd<DM><<<nblk, 32, smem, st>>>(D(p.cst), p.Sc, tstride(), Tn, D(p.K), keep, Pkf, t0, t1);
      LQGK_LAUNCH_CHECK();
    }
    return LQGK_OK;
  }
  // Covariance pass, t up over [t0, t1): the per-trial records; VJP: also the adjoint's linearisation points.
  int cov_fwd(cudaStream_t st, int t0, int t1) const {
    double *Cs = vjp ? D(p.Cs) : nullptr, *J0 = vjp ? D(p.J0) : nullptr;
    float *FU = vjp ? F(p.FU) : nullptr, *JS = vjp ? F(p.JS) : nullptr;
    int rc;
    if (warp_cov) {
      const size_t smem = BigW<DM>::smem_fwd();
      if ((rc = set_smem<DM>((const void*)kw_cov_fwd<DM, !BIG>, smem))) return rc;
      ProfScope ps_(PK_COV_FWD, st);
      kw_cov_fwd<DM, !BIG><<<wblk, WTHR, smem, st>>>(D(p.cst), p.Sc, npad, Tn, D(p.L), D(p.K), vjp, Cs, FU, JS, J0, F(p.rec), t0, t1);
      LQGK_LAUNCH_CHECK();
    } else if constexpr (!BIG) {
      const size_t smem = smem_cov_fwd<DM>();
      if ((rc = set_smem<DM>((const void*)k_cov_fwd<DM>, smem))) return rc;
      ProfScope ps_(PK_COV_FWD, st);
      k_cov_fwd<DM><<<nblk, 32, smem, st>>>(D(p.cst), p.Sc, tstride(), Tn, D(p.L), D(p.K), vjp, Cs, FU, JS, J0, F(p.rec), t0, t1);
      LQGK_LAUNCH_CHECK();
    }
    return LQGK_OK;
  }
  // Observations of the chunk in the per-trial kernels' component-major layout (k_repack_obs): one data set shared by all
  // samples (x_sample_stride == 0) or one per sample of the chunk.
  int repack_obs(cudaStream_t st) {
    const LqgkDims& d = *c.dims;
    const int row = 32 * rt(), nb = (N + row - 1) / row;
    const bool per_sample = d.x_sample_stride != 0;
    const size_t per = (size_t)(Tn + 1) * nb * d.d * row;
    const int nsets = per_sample ? n : 1;
    xcs = per_sample ? per : 0;
    const size_t total = per * nsets;
    const unsigned blocks = (unsigned)std::min<size_t>((total + 255) / 256, (size_t)sm_count() * 16);
    ProfScope ps_(PK_PACK, st);
    k_repack_obs<float><<<blocks, 256, 0, st>>>(c.x_tm, (size_t)d.x_sample_stride, per_sample ? (int)s0 : 0, nsets, N, row, Tn + 1, d.d,
                                                F(p.xc));
    LQGK_LAUNCH_CHECK();
    return LQGK_OK;
  }
  // Per-trial likelihood over the checkpoint segments [ka, kb).  VJP: stores the checkpoints of the carried state.
  int trial_fwd(cudaStream_t st, int ka, int kb) const {
    int rc = LQGK_E_UNSUPPORTED;
    static_for<1, trial_rt_max<DM>() + 1>([&](auto RTC) {
      if (rt() == decltype(RTC)::value)
        rc = launch_trial_fwd<DM, decltype(RTC)::value>(st, F(p.rec), F(p.xc), xcs, n, N, Tn, D(p.ll), vjp ? F(p.hist) : nullptr, ka, kb);
    });
    return rc;
  }
  // Per-trial log-likelihoods out to the caller.  VJP: also the trial weights w (ll_bar; 1 without ll_bar and for the padded
  // samples, whose results are never unpacked).
  int store_ll(cudaStream_t st) const {
    const size_t total = (size_t)n * N, padded = (size_t)npad * N;
    ProfScope ps_(PK_MISC, st);
    k_store_ll<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(D(p.ll), total, (T*)c.ll_out + s0 * N);
    LQGK_LAUNCH_CHECK();
    if (!vjp) return LQGK_OK;
    auto load_w = [&](const T* ll_bar, size_t off, size_t count) -> int {
      k_load_w<T><<<(unsigned)((count + 255) / 256), 256, 0, st>>>(ll_bar, count, F(p.w) + off);
      LQGK_LAUNCH_CHECK();
      return LQGK_OK;
    };
    int rc;
    if ((rc = load_w(c.ll_bar ? (const T*)c.ll_bar + s0 * N : nullptr, 0, total))) return rc;
    return padded > total ? load_w(nullptr, total, padded - total) : LQGK_OK;
  }
  // Zeroes the cotangent accumulators, and (likelihood adjoint) the per-step sums of the padded samples: k_trial_rev never
  // writes those, and the covariance adjoint must read finite data.
  int zero_acc(cudaStream_t st) const {
    if (cudaMemsetAsync(D(p.acc), 0, sizeof(double) * DM::CL.total * p.Sc, st) != cudaSuccess) return LQGK_E_CUDA;
    if (vjp && npad > n &&
        cudaMemsetAsync(F(p.sums) + (size_t)n * Tn * DM::SUMP, 0, sizeof(float) * (size_t)(npad - n) * Tn * DM::SUMP, st) != cudaSuccess)
      return LQGK_E_CUDA;
    return LQGK_OK;
  }
  // Per-trial adjoint over the checkpoint segments [ka, kb), walked downwards: the per-step sums over trials.
  int trial_rev(cudaStream_t st, int ka, int kb) const {
    int rc = LQGK_E_UNSUPPORTED;
    static_for<1, trial_rt_max<DM>() + 1>([&](auto RTC) {
      if (rt() == decltype(RTC)::value)
        rc = launch_trial_rev<DM, decltype(RTC)::value>(st, F(p.rec), F(p.xc), xcs, F(p.hist), F(p.w), n, N, Tn, F(p.sums), F(p.carcb), ka,
                                                        kb);
    });
    return rc;
  }
  // Sequential covariance adjoint, t down over [t0, t1); carC hands its carry from one segment to the next.
  int cov_seq_rev(cudaStream_t st, int t0, int t1) const {
    int rc;
    if (warp_cov) {
      const size_t smem = BigW<DM>::smem_seq();
      if ((rc = set_smem<DM>((const void*)kw_cov_seq_rev<DM>, smem))) return rc;
      ProfScope ps_(PK_COV_REV, st);
      kw_cov_seq_rev<DM><<<wblk, WTHR, smem, st>>>(npad, Tn, N, F(p.w), F(p.FU), F(p.JS), D(p.J0), F(p.sums), F(p.SGB), D(p.SGBI), F(p.SFW), t0,
                                                   t1, D(p.carC));
      LQGK_LAUNCH_CHECK();
    } else if constexpr (!BIG) {
      const size_t smem = smem_cov_seq_rev<DM>();
      if ((rc = set_smem<DM>((const void*)k_cov_seq_rev<DM>, smem))) return rc;
      ProfScope ps_(PK_COV_REV, st);
      k_cov_seq_rev<DM><<<nblk, 32, smem, st>>>(p.Sc, Tn, N, F(p.w), F(p.FU), F(p.JS), D(p.J0), F(p.sums), F(p.SGB), D(p.SGBI), F(p.SFW), t0, t1,
                                                D(p.carC));
      LQGK_LAUNCH_CHECK();
    }
    return LQGK_OK;
  }
  // Time-parallel contraction of the adjoint over [t0, t1), cut into grid.y time ranges: the cotangent accumulators, Lbar, Kbar.
  int contraction(cudaStream_t st, int t0, int t1) const {
    const int len = t1 - t0;
    int rc;
    ProfScope ps_(PK_COV_CONTRIB, st);
    if (warp_cov) {
      // enough (sample x range) warps to put ~12 on every SM when there are few samples
      const int chunks = std::max(1, std::min((len + 3) / 4, (sm_count() * 12 + npad - 1) / npad));
      const size_t smem = BigW<DM>::smem_con();
      if ((rc = set_smem<DM>((const void*)kw_cov_contrib<DM, !BIG>, smem))) return rc;
      kw_cov_contrib<DM, !BIG><<<dim3(wblk, chunks), WTHR, smem, st>>>(D(p.cst), p.Sc, npad, Tn, D(p.L), D(p.K), D(p.Cs), F(p.SGB), D(p.SGBI),
                                                                      F(p.SFW), F(p.sums), D(p.acc), D(p.Lbar), D(p.Kbar), D(p.KbarF), t0, t1);
      LQGK_LAUNCH_CHECK();
    } else if constexpr (!BIG) {
      // (sample-group x time-range) warps: enough to occupy every SM a few times over
      const int cwarps = g_contrib_warps > 0 ? g_contrib_warps : sm_count() * 30;
      const dim3 grid(nblk, std::max(1, std::min((len + 7) / 8, (cwarps + nblk - 1) / nblk)));
      auto pass = [&](auto P) -> int {
        constexpr int PASS = decltype(P)::value;
        const size_t smem = smem_cov_contrib<DM, PASS>();
        if (int rcs = set_smem<DM>((const void*)k_cov_contrib<DM, PASS>, smem)) return rcs;
        k_cov_contrib<DM, PASS><<<grid, 32, smem, st>>>(D(p.cst), p.Sc, Tn, D(p.L), D(p.K), D(p.Cs), F(p.SGB), D(p.SGBI), F(p.SFW), F(p.sums),
                                                        D(p.acc), D(p.Lbar), D(p.Kbar), D(p.KbarF), t0, t1);
        LQGK_LAUNCH_CHECK();
        return LQGK_OK;
      };
      if constexpr (contrib_merged<DM>()) return pass(std::integral_constant<int, 2>{});   // both passes in one kernel
      else if ((rc = pass(std::integral_constant<int, 0>{}))) return rc;
      else return pass(std::integral_constant<int, 1>{});
    }
    return LQGK_OK;
  }
  // Kalman-gain adjoint, t down over [t0, t1); carP hands its carry from one segment to the next.
  int kf_rev(cudaStream_t st, int t0, int t1) const {
    int rc;
    if constexpr (BIG) {
      const size_t smem = BigG<DM>::smem_kf();
      if ((rc = set_smem<DM>((const void*)kw_kf_rev<DM>, smem))) return rc;
      ProfScope ps_(PK_KF_REV, st);
      kw_kf_rev<DM><<<wblk, WTHR, smem, st>>>(D(p.cst), p.Sc, npad, Tn, D(p.Pkf), D(p.Kbar), D(p.acc));
      LQGK_LAUNCH_CHECK();
    } else {
      const size_t smem = smem_kf_rev<DM>();
      if ((rc = set_smem<DM>((const void*)k_kf_rev<DM>, smem))) return rc;
      ProfScope ps_(PK_KF_REV, st);
      k_kf_rev<DM><<<nblk, 32, smem, st>>>(D(p.cst), p.Sc, Tn, D(p.Pkf), D(p.Kbar), D(p.KbarF), D(p.acc), t0, t1, D(p.carP));
      LQGK_LAUNCH_CHECK();
    }
    return LQGK_OK;
  }
  // Riccati adjoint, t up; needs Lbar complete.
  int lqr_rev(cudaStream_t st) const {
    int rc;
    if constexpr (BIG) {
      const size_t smem = BigG<DM>::smem_lqr();
      if ((rc = set_smem<DM>((const void*)kw_lqr_rev<DM>, smem))) return rc;
      ProfScope ps_(PK_LQR_REV, st);
      kw_lqr_rev<DM><<<wblk, WTHR, smem, st>>>(D(p.cst), p.Sc, npad, Tn, c.eps, D(p.L), D(p.Sric), D(p.Lbar), D(p.acc));
      LQGK_LAUNCH_CHECK();
    } else {
      const size_t smem = smem_lqr_rev<DM>();
      if ((rc = set_smem<DM>((const void*)k_lqr_rev<DM>, smem))) return rc;
      ProfScope ps_(PK_LQR_REV, st);
      k_lqr_rev<DM><<<nblk, 32, smem, st>>>(D(p.cst), p.Sc, Tn, c.eps, D(p.L), D(p.Sric), D(p.Lbar), D(p.acc));
      LQGK_LAUNCH_CHECK();
    }
    return LQGK_OK;
  }
  // Cotangent accumulators -> the caller's gradient structs (the actor's only when the call has no dynamics spec).
  int unpack(cudaStream_t st) const {
    UnpackArgs<T> ua{};
    ua.act = *c.act; ua.sigma0 = c.sigma0 ? *c.sigma0 : LqgkMat{nullptr, 0, 0};
    if (c.dyn) ua.dyn = *c.dyn;
    if (c.gact) ua.gact = *c.gact;
    if (c.gdyn) ua.gdyn = *c.gdyn;
    if (c.gsig0) ua.gsigma0 = *c.gsig0;
    ua.x = DM::X; ua.b = DM::B; ua.u = DM::U; ua.y = DM::Y;
    ProfScope ps_(PK_UNPACK, st);
    if (c.dyn) k_unpack<T><<<(n + 63) / 64, 64, 0, st>>>(ua, (int)s0, n, D(p.acc), D(p.cst), p.Sc);
    else k_unpack_actor<T><<<(n + 63) / 64, 64, 0, st>>>(ua, (int)s0, n, D(p.acc), D(p.cst), p.Sc);
    LQGK_LAUNCH_CHECK();
    return LQGK_OK;
  }
  // The caller's cotangents of the gains [s][t][E] -> the workspace array at `off` that the matching adjoint sweep reads
  // (sample-minor for the small systems, sample-major for the large ones).
  int load_gains_bar(cudaStream_t st, size_t off, int E, const void* in) const {
    const size_t total = (size_t)npad * Tn * E;
    ProfScope ps_(PK_MISC, st);
    k_load_rows<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>((const T*)in + s0 * Tn * E, p.Sc, n, npad, Tn, E, !BIG, D(off));
    LQGK_LAUNCH_CHECK();
    return LQGK_OK;
  }
  // Gains [t][E] per sample out to the caller: a transposing copy of the sample-minor workspace arrays of the small systems,
  // a plain copy of the sample-major ones of the large systems.
  int store_gains(cudaStream_t st, size_t off, int E, void* out) const {
    if (!out) return LQGK_OK;
    const size_t total = (size_t)n * Tn * E;
    if constexpr (BIG)
      k_store_ll<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(D(off), total, (T*)out + s0 * Tn * E);
    else
      k_store_rows<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(D(off), p.Sc, n, Tn, E, (T*)out + s0 * Tn * E);
    LQGK_LAUNCH_CHECK();
    return LQGK_OK;
  }
  // Full predictive moments (conditional_moments / belief_tracking_distribution), small systems only: thread-per-sample
  // covariance kernel writing Sigma in the caller's layout, thread-per-trial mean kernel.
  int moments(cudaStream_t st) const {
    if constexpr (BIG) {
      return LQGK_E_UNSUPPORTED;
    } else {
      {
        size_t smem = sizeof(double) * 32 * CovC<DM>::n;
        ProfScope ps_(PK_COV_FWD, st);
        k_cov_moments<DM, T><<<nblk, 32, smem, st>>>(D(p.cst), p.Sc, tstride(), Tn, n, D(p.L), D(p.K), F(p.rec),
                                                     c.Sig_out ? (T*)c.Sig_out + s0 * Tn * DM::N * DM::N : nullptr);
        LQGK_LAUNCH_CHECK();
      }
      if (c.mu_out) {
        size_t total = (size_t)n * N;
        ProfScope ps_(PK_TRIAL_FWD, st);
        k_trial_moments<DM, T><<<(unsigned)((total + 127) / 128), 128, 0, st>>>(F(p.rec), c.x_tm, (size_t)c.dims->x_sample_stride, (int)s0, n,
                                                                              N, Tn, (T*)c.mu_out + s0 * N * Tn * DM::N);
        LQGK_LAUNCH_CHECK();
      }
      return LQGK_OK;
    }
  }
};

template <class DM, class T>
int run(const Call& c) {
  const LqgkDims& d = *c.dims;
  const bool has_dyn = c.dyn != nullptr;
  const bool tv = spec_time_varying(*c.act, true) || (has_dyn && spec_time_varying(*c.dyn, false));
  if (!kernels_cover(c, tv, is_big<DM>())) return LQGK_E_UNSUPPORTED;
  if (!c.ws || ((uintptr_t)c.ws % ALIGN) != 0) return LQGK_E_INVALID;
  // slices: ns concurrent streams, each with its own workspace part and chunk size Sc
  int ns = gains_mode(c.mode) ? 1 : std::max(1, std::min(g_streams, (int)((d.S + 31) / 32)));
  size_t Sc = 0;
  for (; ns >= 1; --ns) {
    const int32_t want = (int32_t)up(((size_t)d.S + ns - 1) / ns, 32);
    Sc = choose_chunk<DM>(d, c.mode, tv, c.ws_bytes / ns / ALIGN * ALIGN, want);
    if (Sc > 0) break;
  }
  if (Sc == 0) return LQGK_E_WORKSPACE;
  const Plan p = make_plan<DM>(d, c.mode, tv, Sc);
  const size_t slice_bytes = up(p.bytes, ALIGN);
  const int Tn = d.T, N = d.N;
  const bool vjp = c.mode == LQGK_MODE_VJP;
  // time segments of the launch sequence of a chunk of n samples (see below)
  auto segments = [&](int n) {
    if (is_big<DM>() || !vjp || g_aux_streams == 0 || n > g_pipe_max_samples) return 1;
    return std::max(1, std::min(g_pipe_segments, trial_geom<DM>(N, Tn).nseg));
  };
  const bool pipelined = segments((int)((size_t)d.S - ((size_t)d.S - 1) / Sc * Sc)) > 1;   // (the last chunk is the smallest)
  const int nstreams = (ns > 1 ? ns : 0) + (pipelined ? 3 * ns : 0);
  if (nstreams > 0) {
    if (int rcp = g_pool.acquire(nstreams, c.stream)) return rcp;
  }
  const int aux0 = ns > 1 ? ns : 0;     // index of the first auxiliary stream
  // internal streams this call has forked work onto (only those are joined back: under CUDA-graph capture a stream that was
  // never forked from the caller's stream is not part of the capture and must not be waited on)
  uint64_t touched = 0;
  auto touch = [&](cudaStream_t s) {
    for (int i = 0; i < nstreams; ++i)
      if (g_pool.streams[i] == s) touched |= 1ull << i;
  };
  // make `to` wait for everything enqueued on `from` so far
  auto is_idle_pool_stream = [&](cudaStream_t s) {
    for (int i = 0; i < nstreams; ++i)
      if (g_pool.streams[i] == s) return ((touched >> i) & 1ull) == 0;
    return false;
  };
  auto dep = [&](cudaStream_t from, cudaStream_t to) {
    if (from == to) return;
    if (is_idle_pool_stream(from)) return;   // nothing of this call runs there (and under capture it is outside the graph)
    cudaEvent_t e = g_pool.next_event();
    cudaEventRecord(e, from);
    cudaStreamWaitEvent(to, e, 0);
    touch(to);
  };
  if (ns > 1) {
    if (cudaEventRecord(g_pool.fork, c.stream) != cudaSuccess) return LQGK_E_CUDA;
    for (int i = 0; i < ns; ++i) {
      if (cudaStreamWaitEvent(g_pool.streams[i], g_pool.fork, 0) != cudaSuccess) return LQGK_E_CUDA;
      touched |= 1ull << i;
    }
  }
  // join on every exit path once side streams may have work
  struct Joiner {
    int nstreams;
    cudaStream_t main;
    const uint64_t* touched;
    ~Joiner() {
      // slice streams (and, on error paths, auxiliary streams) rejoin the caller's stream
      for (int i = 0; i < nstreams; ++i) {
        if (!((*touched >> i) & 1ull)) continue;
        cudaEventRecord(g_pool.joins[i], g_pool.streams[i]);
        cudaStreamWaitEvent(main, g_pool.joins[i], 0);
      }
    }
  } joiner{nstreams, c.stream, &touched};

  int chunk_idx = 0;
  for (size_t s0 = 0; s0 < (size_t)d.S; s0 += Sc, ++chunk_idx) {
    const int n = (int)std::min(Sc, (size_t)d.S - s0);
    const int npad = (int)up(n, 32);
    cudaStream_t st = c.stream;
    char* base = (char*)c.ws;
    if (ns > 1) {
      st = g_pool.streams[chunk_idx % ns];
      base += (size_t)(chunk_idx % ns) * slice_bytes;
    }
    const bool warp_cov = is_big<DM>() || (!tv && d.S <= g_warp_cov_max_samples);
    const bool keep = vjp || c.mode == LQGK_MODE_GAINS_VJP;
    Chunk<DM, T> k{c, p, base, s0, n, npad, npad / 32, (npad + BW_WARPS - 1) / BW_WARPS, Tn, N, tv, vjp, keep, warp_cov};
    int rc;
    if ((rc = k.pack(st))) return rc;
    if (c.mode == LQGK_MODE_GAINS) {
      if (c.L_out) {
        if ((rc = k.template lqr_fwd<true>(st))) return rc;
        if ((rc = k.store_gains(st, p.L, DM::EL, c.L_out))) return rc;
        if ((rc = k.store_gains(st, p.l, DM::U, c.l_out))) return rc;
        if ((rc = k.store_gains(st, p.H, DM::U * DM::U, c.H_out))) return rc;
      }
      if (c.K_out) {
        if ((rc = k.kf_fwd(st, 0, Tn))) return rc;
        if ((rc = k.store_gains(st, p.K, DM::EK, c.K_out))) return rc;
      }
      continue;
    }
    if (c.mode == LQGK_MODE_GAINS_VJP) {
      // both sweeps again, keeping S_t / P_t, then their adjoints from the caller's cotangents; a NULL cotangent skips its pair
      if ((rc = k.zero_acc(st))) return rc;
      if (c.L_bar) {
        if ((rc = k.template lqr_fwd<false>(st))) return rc;
        if ((rc = k.load_gains_bar(st, p.Lbar, DM::EL, c.L_bar))) return rc;
        if ((rc = k.lqr_rev(st))) return rc;
      }
      if (c.K_bar) {
        if ((rc = k.kf_fwd(st, 0, Tn))) return rc;
        if ((rc = k.load_gains_bar(st, p.Kbar, DM::EK, c.K_bar))) return rc;
        // the Kalman adjoint of the small systems adds a second cotangent part, which only the likelihood's contraction fills
        if (!is_big<DM>() && cudaMemsetAsync(k.D(p.KbarF), 0, sizeof(double) * Tn * DM::EK * p.Sc, st) != cudaSuccess) return LQGK_E_CUDA;
        if ((rc = k.kf_rev(st, 0, Tn))) return rc;
      }
      if ((rc = k.unpack(st))) return rc;
      continue;
    }
    if (c.mode == LQGK_MODE_MOMENTS) {
      if ((rc = k.template lqr_fwd<false>(st))) return rc;
      if ((rc = k.kf_fwd(st, 0, Tn))) return rc;
      if ((rc = k.moments(st))) return rc;
      continue;
    }
    // Launch sequence of the likelihood and its adjoint.  Few samples: every sweep over time is latency-bound (T dependent
    // steps, ~1-2.5 ms each whatever the sample count) and the GPU idles behind the chain of nine sweeps.  The sweeps of one
    // direction are therefore cut into G time segments and run as a software pipeline over the chunk's internal streams
    // x1..x3: segment g of a consumer starts as soon as segment g of its producer is done.
    //   t up  : kf_fwd (x1) -> cov_fwd (x2) -> trial_fwd (st)        [after lqr_fwd, which runs t down and feeds cov_fwd]
    //   t down: trial_rev (st) -> cov_seq_rev (x1) -> contraction (x2) -> kf_rev (x3);  lqr_rev (t up) follows on x2
    // Carries between segments: P_t, C_t and the checkpoints of c_t are stored per step anyway (adjoint linearisation points);
    // the adjoint carries (cb, Cb, Pnb) go through three small buffers.  G = 1 (forward only, large systems, kernel overlap
    // off, chunks above g_pipe_max_samples, T within one checkpoint interval) is the same sequence on the chunk's stream.
    const int G = segments(n);
    cudaStream_t x1 = st, x2 = st, x3 = st;
    if (G > 1) {
      const int a = aux0 + 3 * (chunk_idx % ns);
      x1 = g_pool.streams[a];
      x2 = g_pool.streams[a + 1];
      x3 = g_pool.streams[a + 2];
    }
    const TrialGeom tg = trial_geom<DM>(N, Tn);
    std::vector<int> kb(G + 1), tb(G + 1);   // segment g: checkpoint segments [kb[g], kb[g + 1]), steps [tb[g], tb[g + 1])
    for (int g = 0; g <= G; ++g) { kb[g] = (int)((long long)g * tg.nseg / G); tb[g] = std::min(Tn, kb[g] * tg.CK); }
    dep(st, x1);                                 // pack done -> kf_fwd on x1 beside lqr_fwd on st
    if ((rc = k.template lqr_fwd<false>(st))) return rc;
    dep(st, x2);                                 // L complete -> covariance pass
    if ((rc = k.repack_obs(st))) return rc;
    for (int g = 0; g < G; ++g) {
      if ((rc = k.kf_fwd(x1, tb[g], tb[g + 1]))) return rc;
      dep(x1, x2);
      if ((rc = k.cov_fwd(x2, tb[g], tb[g + 1]))) return rc;
      dep(x2, st);
      if ((rc = k.trial_fwd(st, kb[g], kb[g + 1]))) return rc;
    }
    if ((rc = k.store_ll(st))) return rc;
    if (!vjp) continue;
    if ((rc = k.zero_acc(st))) return rc;
    for (int g = G - 1; g >= 0; --g) {
      if ((rc = k.trial_rev(st, kb[g], kb[g + 1]))) return rc;
      dep(st, x1);
      if ((rc = k.cov_seq_rev(x1, tb[g], tb[g + 1]))) return rc;
      dep(x1, x2);
      if ((rc = k.contraction(x2, tb[g], tb[g + 1]))) return rc;
      dep(x2, x3);
      if ((rc = k.kf_rev(x3, tb[g], tb[g + 1]))) return rc;
    }
    if ((rc = k.lqr_rev(x2))) return rc;         // after every contraction segment (Lbar complete), in order on x2
    dep(x2, st);
    dep(x3, st);
    if ((rc = k.unpack(st))) return rc;
  }
  return LQGK_OK;
}

// The per-trial likelihood under signal-dependent noise, all FP64 (small and FP64-only tuples): one thread per (sample, trial).
template <class DM>
int launch_sdn_loglik(const SdnLikArgs& a, bool f64, cudaStream_t st) {
  const unsigned blocks = (unsigned)(((size_t)a.S * a.N + 63) / 64);
  if (f64) k_sdn_loglik<DM, double><<<blocks, 64, 0, st>>>(a);
  else k_sdn_loglik<DM, float><<<blocks, 64, 0, st>>>(a);
  LQGK_LAUNCH_CHECK();
  return LQGK_OK;
}

// One specialisation per line of LQGK_FOR_EACH_DIMS (defined in lqgk_inst.cu; run_sdn* for joint dims <= 12 only).
template <class DM>
struct Runner {
  static int run_f32(const Call& c);
  static int run_f64(const Call& c);
  static size_t plan_bytes(const LqgkDims& d, int mode, int32_t max_chunk);
  static int run_sdn(const SdnArgs& a, cudaStream_t st);   // signal-dependent-noise gains (b, u, y of this tuple)
  static int run_sdn_loglik(const SdnLikArgs& a, bool f64, cudaStream_t st);   // likelihood under signal-dependent noise
};

}  // namespace lqgk
