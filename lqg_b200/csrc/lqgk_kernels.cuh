// lqgk_kernels.cuh -- __global__ kernels for sm_100a.
//
// Mapping (DESIGN.md section 3):
//  * per-sample FP64 recursions (k_lqr_fwd, k_kf_fwd, k_cov_fwd and their adjoints): ONE THREAD PER PARAMETER
//    SAMPLE, 32 samples per single-warp CTA.  All matrices live in registers as statically indexed arrays, the
//    per-sample derived constants and cotangent accumulators in shared memory laid out [element][lane] (bank =
//    lane, conflict free).  Per-step state is exchanged through HBM workspace arrays laid out sample-minor
//    [t][element][sample] so every warp access is one coalesced 256-byte line.
//  * per-trial FP32 recursions (k_trial_fwd, k_trial_rev): ONE WARP PER SAMPLE, LANE = TRIAL (RT trials per lane).
//    The per-step operator records of the sample ([t][REC] floats, contiguous) are staged into shared memory by
//    the TMA engine with 1-D bulk async copies (cp.async.bulk + mbarrier complete_tx) in a per-warp ring, and
//    read as warp-wide broadcasts.  Observations are time-major so lane=trial loads are coalesced.
#pragma once
#include <cuda_runtime.h>

#include "lqgk_core.h"
#include "lqgk_pack.h"
#include "lqgk_stages.h"

namespace lqgk {

constexpr unsigned FULL = 0xffffffffu;

// ------------------------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// 1-D bulk async copy global -> shared through the TMA engine (SASS: UBLKCP), completion on an mbarrier.
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// 1-D bulk async copy shared -> global (TMA store, bulk-group completion).
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// Per-thread asynchronous global->shared copies (LDGSTS) used as a register-free software prefetch.
template <int BYTES>
__device__ __forceinline__ void cp_async(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_u32(dst)), "l"(src), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// =========================================================================================== boundary kernels
template <class T>
__global__ void k_pack(PackArgs<T> a, int s0, int n_valid, int n_pad, double* cst, size_t Sc, size_t tstride, int nt) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int t = blockIdx.y;
  if (i >= n_pad || t >= nt) return;
  int s = s0 + (i < n_valid ? i : n_valid - 1);   // padding lanes replicate the last valid sample
  WView out{cst + (size_t)t * tstride + i, Sc};
  pack_sample<T>(a, s, t, [&](int e) -> double& { return out(e); });
}

template <class T>
__global__ void k_unpack(UnpackArgs<T> a, int s0, int n_valid, const double* acc, const double* cst, size_t Sc) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_valid) return;
  unpack_sample<T>(a, s0 + i, [&](int e) { return acc[(size_t)e * Sc + i]; }, [&](int e) { return cst[(size_t)e * Sc + i]; });
}

// (k_unpack for the gains adjoint, which has no dynamics spec)
template <class T>
__global__ void k_unpack_actor(UnpackArgs<T> a, int s0, int n_valid, const double* acc, const double* cst, size_t Sc) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_valid) return;
  unpack_sample<T, false>(a, s0 + i, [&](int e) { return acc[(size_t)e * Sc + i]; }, [&](int e) { return cst[(size_t)e * Sc + i]; });
}

// SoA workspace [t][E][Sc] -> user layout [s][t][E]
template <class T>
__global__ void k_store_rows(const double* ws, size_t Sc, int n_valid, int Tn, int E, T* out /* already offset by s0 */) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t total = (size_t)n_valid * Tn * E;
  if (idx >= total) return;
  int e = idx % E;
  int t = (idx / E) % Tn;
  int s = idx / ((size_t)E * Tn);
  out[idx] = (T)ws[((size_t)t * E + e) * Sc + s];
}
// The reverse of k_store_rows / k_store_ll for the cotangents of the gains: user layout [s][t][E] -> FP64 workspace, sample-minor
// [t][E][Sc] (small systems) or sample-major [s][t][E] (large systems); the padded samples n_valid <= s < n_pad get zeros.
template <class T>
__global__ void k_load_rows(const T* in /* already offset by s0 */, size_t Sc, int n_valid, int n_pad, int Tn, int E, bool sample_minor,
                            double* ws) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t total = (size_t)n_pad * Tn * E;
  if (idx >= total) return;
  int e = idx % E;
  int t = (idx / E) % Tn;
  int s = idx / ((size_t)E * Tn);
  ws[sample_minor ? ((size_t)t * E + e) * Sc + s : idx] = s < n_valid ? (double)in[idx] : 0.0;
}
template <class T>
__global__ void k_store_ll(const double* ll_ws, size_t count, T* out) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < count) out[idx] = (T)ll_ws[idx];
}
template <class T>
__global__ void k_load_w(const T* ll_bar /* nullable, already offset */, size_t count, float* w) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < count) w[idx] = ll_bar ? (float)ll_bar[idx] : 1.f;
}
template <class T>
__global__ void k_pack_obs(int N, int T1, int d, const T* x, float* x_tm) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t total = (size_t)N * T1 * d;
  if (idx >= total) return;
  int k = idx % d;
  int i = (idx / d) % N;
  int t = idx / ((size_t)d * N);
  x_tm[idx] = (float)x[((size_t)i * T1 + t) * d + k];
}

// Observations for the per-trial kernels: x_tm[(s)][T+1][N][d] (ABI layout, trial-major inside a step) -> blocked and
// component-major xc[(s)][T+1][NB][d][ROW]: the trials are cut into NB blocks of ROW = 32 * RT (one block per pass of the
// per-trial kernels, RT trials per lane), and inside a block every component is one contiguous row.  A lane's pair of
// ADJACENT trials (2i, 2i+1) of one component is then one aligned 64-bit element = one f32x2 register pair (the trial-major
// layout cost ~100 register moves per step in the adjoint kernel to pair the trials up), and all of a lane's elements of a
// step sit at compile-time offsets from one pointer.  Columns beyond the last trial repeat it (finite; masked by weight 0).
template <class T>   // (a template only so that the header can be included from several translation units)
__global__ void k_repack_obs(const T* __restrict__ x_tm, size_t x_sample_stride, int s_first, int nsets, int N, int row, int T1, int d,
                             float* __restrict__ xc) {
  const int nb = (N + row - 1) / row;
  const size_t per = (size_t)T1 * nb * d * row;
  const size_t total = per * nsets;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int col = idx % row;
    const int m = (idx / row) % d;
    const int blk = (idx / ((size_t)row * d)) % nb;
    const int t = (idx / ((size_t)row * d * nb)) % T1;
    const size_t ds = idx / per;
    const int i = blk * row + col;
    const int ic = i < N ? i : N - 1;
    xc[idx] = x_tm[(size_t)(s_first + ds) * x_sample_stride + ((size_t)t * N + ic) * d + m];
  }
}

// =========================================================================================== per-sample kernels
// All launched with blockDim = 32 and gridDim = Sc / 32 (Sc is padded to a multiple of 32 by k_pack).
template <class DM, bool AFFINE>
__global__ void __launch_bounds__(32) k_lqr_fwd(const double* cst, size_t Sc, size_t tstride, int Tn, double eps, double* L,
                                                int save_S, double* Sric, double* l, double* H) {
  extern __shared__ __align__(16) double sm[];
  const int lane = threadIdx.x;
  const size_t s = (size_t)blockIdx.x * 32 + lane;
  lqr_fwd_body<DM, AFFINE>(GCst{cst + s, Sc, tstride}, WView{sm + lane, 32}, Tn, eps, WView{L + s, Sc}, save_S != 0,
                           WView{Sric + s, Sc}, WView{l + s, Sc}, WView{H + s, Sc});
}

template <class DM>
__global__ void __launch_bounds__(32) k_kf_fwd(const double* cst, size_t Sc, size_t tstride, int Tn, double* K, int save_P,
                                               double* Pkf, int t0, int t1) {
  extern __shared__ __align__(16) double sm[];
  const int lane = threadIdx.x;
  const size_t s = (size_t)blockIdx.x * 32 + lane;
  kf_fwd_body<DM>(GCst{cst + s, Sc, tstride}, WView{sm + lane, 32}, Tn, WView{K + s, Sc}, save_P != 0, WView{Pkf + s, Sc}, t0, t1);
}

template <class KC, class La>
__device__ __forceinline__ void flush_acc_atomic(double* g, size_t stride, const La& l, int nseg) {
  for (int i = 0; i < nseg; ++i) {
    int go, lo, len;
    KC::seg(i, go, lo, len);
    for (int e = 0; e < len; ++e) atomicAdd(&g[(size_t)(go + e) * stride], l(lo + e));
  }
}

// ------------------------------------------------------------------------------------------- step-input ring
// The sequential per-sample kernels are latency-bound if each step's inputs are fetched with ordinary loads (one
// HBM round trip per dependent phase, ~1 warp per scheduler).  Instead each warp keeps a ring of NST "step input"
// stages in shared memory that the TMA engine fills ahead of time: for a warp's 32 consecutive samples, row e of
// step t of a sample-minor array is one contiguous 256-byte line, copied with one cp.async.bulk issued by lane
// (e mod 32); an optional float source copies one [CNTF]-float row per sample (lane = sample) from the
// sample-major sums array.  The stage layout is [row][32 lanes] doubles (lane-strided, bank-conflict free).
// Adjoint linearisation points that are written once and read once (Fu_t, (J_t, S'^-1_t), Sgb_t, SF_t) are stored in FP32: they
// enter every adjoint step linearly (no accumulation of their rounding over time; measured: no change of any gradient error, see
// DESIGN.md) and were 56 % of the FP64 workspace traffic of the per-sample kernels, two of which run at 70-90 % of HBM bandwidth.
using lin_t = float;
struct RingSrc {
  const void* base;     // array base + first sample of the warp
  int rows;             // rows (elements) per time step
  int f32;              // 0: rows of 32 doubles (256 B), 1: rows of 32 floats (128 B)
};
struct FView {
  const float* p;
  __device__ __forceinline__ double operator()(int e) const { return (double)p[(size_t)e * 32]; }
};
// Offsets inside a stage are counted in 128-byte units: a double row takes 2, a float row 1.
template <int NSRC, int NST>
struct StepRing {
  RingSrc src[NSRC];
  size_t Sc;
  const float* fsrc;    // optional: sums + s0 * Tn * SUMP + LO   (nullptr = none)
  int frow_stride;      // Tn * SUMP (floats between consecutive samples)
  int fstep_stride;     // SUMP
  int fcnt;             // floats per row copy (multiple of 4)
  double* buf;          // [NST][stage_doubles]
  uint64_t* bars;       // [NST]
  int lane, total_units, stage_doubles;
  uint32_t phase_bits;

  __host__ __device__ __forceinline__ static constexpr int stage_size(int total_units, int fcnt) { return total_units * 16 + (32 * fcnt + 1) / 2; }
  __device__ __forceinline__ void init() {
    if (lane == 0) {
      for (int i = 0; i < NST; ++i) mbar_init(&bars[i], 1);
      fence_mbar_init();
    }
    phase_bits = 0;
    __syncwarp();
  }
  // Caller guarantees (by __syncwarp) that no lane still reads stage `st`.
  __device__ __forceinline__ void issue(int t, int st) {
    char* dst = reinterpret_cast<char*>(buf + (size_t)st * stage_doubles);
    fence_proxy_async();
    if (lane == 0) mbar_expect_tx(&bars[st], (uint32_t)(total_units * 128 + (fsrc ? 32 * fcnt * 4 : 0)));
    int unit = 0;
    LQGK_UNROLL for (int i = 0; i < NSRC; ++i) {
      const int u = src[i].f32 ? 1 : 2;
      for (int r = lane; r < src[i].rows; r += 32)
        bulk_g2s(dst + (size_t)(unit + r * u) * 128, reinterpret_cast<const char*>(src[i].base) + ((size_t)t * src[i].rows + r) * Sc * (u * 4),
                 (uint32_t)u * 128, &bars[st]);
      unit += src[i].rows * u;
    }
    if (fsrc) {
      float* fdst = reinterpret_cast<float*>(dst + (size_t)total_units * 128);
      bulk_g2s(fdst + lane * fcnt, fsrc + (size_t)lane * frow_stride + (size_t)t * fstep_stride, (uint32_t)fcnt * 4, &bars[st]);
    }
  }
  __device__ __forceinline__ const double* wait(int st) {
    mbar_wait(&bars[st], (phase_bits >> st) & 1u);
    phase_bits ^= (1u << st);
    return buf + (size_t)st * stage_doubles;
  }
  // this lane's view of a double source that starts `unit_off` units into the stage
  __device__ __forceinline__ WView view(const double* stage, int unit_off) const {
    return WView{const_cast<double*>(stage) + (size_t)unit_off * 16 + lane, 32};
  }
  // ... and of a float source
  __device__ __forceinline__ FView fview(const double* stage, int unit_off) const {
    return FView{reinterpret_cast<const float*>(stage + (size_t)unit_off * 16) + lane};
  }
  __device__ __forceinline__ const float* frow(const double* stage) const {
    return reinterpret_cast<const float*>(stage + (size_t)total_units * 16) + lane * fcnt;
  }
};

// Record sink: each lane assembles its sample's record ([REC] floats, one 16-byte-aligned row) in shared memory and
// hands it to the TMA engine: one bulk store per lane and step into rec[sample][t][REC].  Two row buffers alternate so
// the store of step t overlaps the arithmetic of step t+1 (no per-element copy loop, no warp synchronisation).
template <class DM>
struct SmemRecSink {
  static constexpr int RS = DM::REC;          // floats per row
  static constexpr int FLOATS = 2 * 32 * RS;  // two buffers
  float* stage;
  float* gbase;   // rec + (this lane's sample) * Tn * REC
  int lane, buf;
  __device__ __forceinline__ void put(int idx, float v) { stage[(buf * 32 + lane) * RS + idx] = v; }
  __device__ __forceinline__ void commit(int t) {
    fence_proxy_async();                       // my generic-proxy writes -> visible to the async proxy
    bulk_s2g(gbase + (size_t)t * DM::REC, stage + (buf * 32 + lane) * RS, DM::REC * sizeof(float));
    bulk_commit();
    buf ^= 1;
    bulk_wait_read<1>();                       // the buffer about to be rewritten (store of step t-1) has been read
  }
  __device__ __forceinline__ void finish() { bulk_wait<0>(); }
};

constexpr int SEQ_NST = 3;   // ring depth of the sequential kernels

// Covariance pass (forward).  Ring inputs per step: L_t, K_t.
// [t0, t1): time range of this launch; t0 > 0 continues from the C_{t0} an earlier launch saved in Cs (save_adj on).
template <class DM>
__global__ void __launch_bounds__(32) k_cov_fwd(const double* cst, size_t Sc, size_t tstride, int Tn, const double* L,
                                                const double* K, int save_adj, double* Cs, lin_t* FU, lin_t* JS, double* J0,
                                                float* rec, int t0, int t1) {
  extern __shared__ __align__(128) double sm[];
  constexpr int B = DM::B, U = DM::U, Y = DM::Y, R = DM::R, D = DM::D;
  using C = CovC<DM>;
  using SR = CovSeqRev<DM>;
  using Ring = StepRing<2, SEQ_NST>;
  const int lane = threadIdx.x;
  const size_t s0 = (size_t)blockIdx.x * 32, s = s0 + lane;
  constexpr int ROWS = DM::EL + DM::EK;
  double* ring_buf = sm;
  double* lcp = ring_buf + (size_t)SEQ_NST * ROWS * 32;
  float* stage = reinterpret_cast<float*>(lcp + C::n * 32);
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage + SmemRecSink<DM>::FLOATS);
  for (int i = lane; i < SmemRecSink<DM>::FLOATS; i += 32) stage[i] = 0.f;
  __syncwarp();
  Ring ring{{{L + s0, DM::EL, 0}, {K + s0, DM::EK, 0}}, Sc, nullptr, 0, 0, 0, ring_buf, bars, lane, 2 * ROWS, ROWS * 32, 0};
  ring.init();
  for (int k = 0; k < SEQ_NST && t0 + k < t1; ++k) ring.issue(t0 + k, k);
  WView lc{lcp + lane, 32};
  GCst g{cst + s, Sc, tstride};
  load_consts<C>(g.at(tstride ? t0 : 0), lc, C::NSEG);
  SmemRecSink<DM> sink{stage, rec + s * Tn * DM::REC, lane, 0};
  double Cm[R * R];
  if (t0 == 0) {
    double K0[B * Y], J0v[R * D];
    LQGK_UNROLL for (int i = 0; i < B * Y; ++i) K0[i] = K[(size_t)i * Sc + s];
    CovFwd<DM>::init(lc, K0, Cm, J0v);
    if (save_adj) { LQGK_UNROLL for (int i = 0; i < R * D; ++i) J0[(size_t)i * Sc + s] = J0v[i]; }
  } else {
    load_sym_ws<R>(WView{Cs + s, Sc}, (size_t)t0 * DM::EC, Cm);
  }
  // (constants stay in shared memory here: a register copy of the 40 covariance constants made this kernel 10 % slower)
  for (int t = t0; t < t1; ++t) {
    const int st = (t - t0) % SEQ_NST;
    const double* stg = ring.wait(st);
    if (tstride && t != t0) load_consts<C>(g.at(t), lc, C::NSEG);
    double Lt[U * B], Kt[B * Y];
    {
      WView lv = ring.view(stg, 0), kv = ring.view(stg, 2 * DM::EL);
      LQGK_UNROLL for (int i = 0; i < U * B; ++i) Lt[i] = lv(i);
      LQGK_UNROLL for (int i = 0; i < B * Y; ++i) Kt[i] = kv(i);
    }
    __syncwarp();
    if (t + SEQ_NST < t1) ring.issue(t + SEQ_NST, st);
    if (save_adj) store_sym<R>(WView{Cs + s, Sc}, (size_t)t * DM::EC, Cm);
    CovFwd<DM>::step(lc, Lt, Kt, Cm, [&](int idx, float v) { sink.put(idx, v); },
                     [&](int which, int e, double v) {
                       if (save_adj) {
                         if (which == 0) FU[((size_t)t * SR::NSF + e) * Sc + s] = (lin_t)v;
                         else JS[((size_t)t * SR::NJS + e) * Sc + s] = (lin_t)v;
                       }
                     });
    sink.commit(t);
  }
  if (save_adj && t1 < Tn) store_sym<R>(WView{Cs + s, Sc}, (size_t)t1 * DM::EC, Cm);   // where the next time segment continues from
  sink.finish();
}

// ------------------------------------------------------------------------------------------- moments (slow path)
// conditional_moments / belief_tracking_distribution (system.py:142-235, 250-257): the same recursions, emitting the full
// predictive moments instead of the log-density.  Covariances: thread per sample, written straight to the caller's
// Sigma[s][t][n][n]; means: thread per (sample, trial), written to mu[s][i][t][n].  Output-bound by construction (n^2 + N n
// numbers per sample-step), so these kernels use plain loads / stores.
struct DirectRecSink {
  float* row;
  int rec;
  __device__ __forceinline__ void put(int idx, float v) { row[idx] = v; }
  __device__ __forceinline__ void commit(int) { row += rec; }
};
template <class DM, class T>
__global__ void __launch_bounds__(32) k_cov_moments(const double* cst, size_t Sc, size_t tstride, int Tn, int n_valid, const double* L,
                                                    const double* K, float* rec, T* __restrict__ Sig_out) {
  extern __shared__ __align__(16) double sm[];
  const int lane = threadIdx.x;
  const size_t s = (size_t)blockIdx.x * 32 + lane;
  DirectRecSink sink{rec + s * Tn * DM::REC, DM::REC};
  const bool emit = Sig_out != nullptr && s < (size_t)n_valid;
  WView none{nullptr, 0};
  cov_fwd_body<DM>(GCst{cst + s, Sc, tstride}, WView{sm + lane, 32}, Tn, WView{const_cast<double*>(L) + s, Sc},
                   WView{const_cast<double*>(K) + s, Sc}, false, none, none, none, none, sink,
                   [&](int t, int e, double v) { if (emit) Sig_out[((size_t)s * Tn + t) * (DM::N * DM::N) + e] = (T)v; });
}
template <class DM, class T>
__global__ void k_trial_moments(const float* __restrict__ rec, const float* __restrict__ x_all, size_t x_sample_stride, int s_first,
                                int n_samples, int N, int Tn, T* __restrict__ mu_out) {
  constexpr int D = DM::D, R = DM::R, NJ = DM::N;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t s = idx / N;
  const int i = (int)(idx % N);
  if (s >= (size_t)n_samples) return;
  const float* x_tm = x_all + (size_t)(s_first + s) * x_sample_stride;
  float c[R], x0[D], x1[D], mu[NJ];
  LQGK_UNROLL for (int k = 0; k < R; ++k) c[k] = 0.f;
  LQGK_UNROLL for (int k = 0; k < D; ++k) x0[k] = x_tm[(size_t)i * D + k];
  T* out = mu_out + (s * N + i) * (size_t)Tn * NJ;
  for (int t = 0; t < Tn; ++t) {
    LQGK_UNROLL for (int k = 0; k < D; ++k) x1[k] = x_tm[((size_t)(t + 1) * N + i) * D + k];
    Trial<DM>::template moments<float>(rec + (s * Tn + t) * DM::REC, x0, x1, c, mu);
    LQGK_UNROLL for (int k = 0; k < NJ; ++k) out[(size_t)t * NJ + k] = (T)mu[k];
    LQGK_UNROLL for (int k = 0; k < D; ++k) x0[k] = x1[k];
  }
}

// Sequential covariance adjoint: lean (no constants, no accumulators); emits Sgb_t, SF_t for the parallel contraction.
// Ring inputs per step: Fu_t, (J_t, S'^-1_t) and the [SUM_J, SUMP) tail of the trial sums.
// [t0, t1): time range of this launch (walked downwards).  t1 < Tn starts from the cotangent an earlier launch left in
// `carry` ([R*R][Sc]); t0 > 0 leaves its own there instead of finishing with the initial-condition term.
template <class DM>
__global__ void __launch_bounds__(32) k_cov_seq_rev(size_t Sc, int Tn, int N, const float* w, const lin_t* FU, const lin_t* JS,
                                                    const double* J0, const float* sums, lin_t* SGB, double* SGBI, lin_t* SFW,
                                                    int t0, int t1, double* carry) {
  extern __shared__ __align__(128) double sm[];
  using SR = CovSeqRev<DM>;
  using Ring = StepRing<2, SEQ_NST>;
  constexpr int R = DM::R;
  constexpr int UNITS = SR::NSF + SR::NJS, FCNT = DM::SUMP - DM::SUM_J;      // float rows: one 128-byte unit each
  constexpr int STAGE = Ring::stage_size(UNITS, FCNT);
  const int lane = threadIdx.x;
  const size_t s0 = (size_t)blockIdx.x * 32, s = s0 + lane;
  double* scp = sm + (size_t)SEQ_NST * STAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(scp + SR::SC_N * 32);
  Ring ring{{{FU + s0, SR::NSF, 1}, {JS + s0, SR::NJS, 1}}, Sc, sums + s0 * Tn * DM::SUMP + DM::SUM_J, Tn * DM::SUMP, DM::SUMP, FCNT,
            sm, bars, lane, UNITS, STAGE, 0};
  ring.init();
  const int nsteps = t1 - t0;
  for (int k = 0; k < SEQ_NST && k < nsteps; ++k) ring.issue(t1 - 1 - k, k);
  double sw = 0.0;
  for (int i = 0; i < N; ++i) sw += (double)w[s * N + i];
  WView sc{scp + lane, 32};
  double Cb[R * R];
  if (t1 == Tn) { LQGK_UNROLL for (int i = 0; i < R * R; ++i) Cb[i] = 0.0; }
  else { LQGK_UNROLL for (int i = 0; i < R * R; ++i) Cb[i] = carry[(size_t)i * Sc + s]; }
  for (int kk = 0; kk < nsteps; ++kk) {
    const int t = t1 - 1 - kk, st = kk % SEQ_NST;
    const double* stg = ring.wait(st);
    FView fuv = ring.fview(stg, 0), jsv = ring.fview(stg, SR::NSF);
    const float* fr = ring.frow(stg);
    SR::step([&](int e) { return fuv(e); }, [&](int e) { return jsv(e); }, [&](int idx) { return fr[idx - DM::SUM_J]; }, sw, sc, Cb,
             [&](int e, double v) { SGB[((size_t)t * SR::NSGB + e) * Sc + s] = (lin_t)v; },
             [&](int e, double v) { SFW[((size_t)t * SR::NSF + e) * Sc + s] = (lin_t)v; });
    __syncwarp();
    if (kk + SEQ_NST < nsteps) ring.issue(t1 - 1 - (kk + SEQ_NST), st);
  }
  if (t0 == 0) SR::init([&](int e) { return J0[(size_t)e * Sc + s]; }, Cb, [&](int e, double v) { SGBI[(size_t)e * Sc + s] = v; });
  else { LQGK_UNROLL for (int i = 0; i < R * R; ++i) carry[(size_t)i * Sc + s] = Cb[i]; }
}

// Time-parallel contraction.  grid = (Sc / 32, chunks), block = one warp owning a contiguous range of time steps of
// its 32 samples.  Ring inputs per step: L_t, K_t, C_t, SF_t (, Sgb_t) and the trial sums F-block.  The contributions
// to the derived-constant cotangents are accumulated over the warp's time range in shared memory ([element][lane])
// and added to the global accumulators with one atomicAdd per element at the end.
// PASS 0 / 1: the two register-limited halves (run concurrently on two streams); PASS 2: both in one kernel (small systems).
template <class DM>
__host__ __device__ constexpr bool contrib_merged() { return DM::N <= 6; }
// ring depth of the contraction kernels: 2 stages when they fit in shared memory beside the constants, else 1
template <class DM, int PASS>
__host__ __device__ constexpr int contrib_nst() {
  using SR = CovSeqRev<DM>;
  constexpr int UNITS = 2 * (DM::EL + DM::EK + DM::EC) + SR::NSF + (PASS != 1 ? SR::NSGB : 0);
  constexpr size_t two = sizeof(double) * ((size_t)2 * (UNITS * 16 + 16 * DM::SUM_J) + 2 * CovC<DM>::n * 32);
  return two <= 200 * 1024 ? 2 : 1;
}
template <class DM, int PASS>
__global__ void __launch_bounds__(32) k_cov_contrib(const double* cst, size_t Sc, int Tn, const double* L, const double* K,
                                                    const double* Cs, const lin_t* SGB, const double* SGBI, const lin_t* SFW,
                                                    const float* sums, double* acc, double* Lbar, double* Kbar, double* KbarF,
                                                    int ta, int tb) {
  extern __shared__ __align__(128) double sm[];
  constexpr int B = DM::B, U = DM::U, Y = DM::Y, R = DM::R;
  using SR = CovSeqRev<DM>;
  using CC = CovContrib<DM>;
  using C = CovC<DM>;
  constexpr bool P0 = PASS == 0 || PASS == 2, P1 = PASS == 1 || PASS == 2;
  constexpr int NSRC = P0 ? 5 : 4;
  constexpr int PAR_NST = contrib_nst<DM, PASS>();
  using Ring = StepRing<NSRC, PAR_NST>;
  constexpr int UNITS = 2 * (DM::EL + DM::EK + DM::EC) + SR::NSF + (P0 ? SR::NSGB : 0);   // 128-byte units (double rows: 2, float rows: 1)
  constexpr int FCNT = DM::SUM_J;   // = round4(N*N)
  constexpr int STAGE = Ring::stage_size(UNITS, FCNT);
  const int lane = threadIdx.x;
  const size_t s0 = (size_t)blockIdx.x * 32, s = s0 + lane;
  double* lcp = sm + (size_t)PAR_NST * STAGE;
  double* lap = lcp + C::n * 32;
  uint64_t* bars = reinterpret_cast<uint64_t*>(lap + C::n * 32);
  const int nq = gridDim.y, q = blockIdx.y;       // the launch covers [ta, tb), cut into nq time ranges
  const int per = (tb - ta + nq - 1) / nq;
  const int t0 = min(tb, ta + q * per), t1 = min(tb, t0 + per);
  if (t0 >= t1) return;
  Ring ring;
  ring.src[0] = {L + s0, DM::EL, 0};
  ring.src[1] = {K + s0, DM::EK, 0};
  ring.src[2] = {Cs + s0, DM::EC, 0};
  ring.src[3] = {SFW + s0, SR::NSF, 1};
  if constexpr (P0) ring.src[4] = {SGB + s0, SR::NSGB, 1};
  ring.Sc = Sc; ring.fsrc = sums + s0 * Tn * DM::SUMP; ring.frow_stride = Tn * DM::SUMP; ring.fstep_stride = DM::SUMP;
  ring.fcnt = FCNT; ring.buf = sm; ring.bars = bars; ring.lane = lane; ring.total_units = UNITS; ring.stage_doubles = STAGE;
  ring.init();
  for (int k = 0; k < PAR_NST && t0 + k < t1; ++k) ring.issue(t0 + k, k);
  WView lc{lcp + lane, 32}, la{lap + lane, 32};
  load_consts<C>(WView{const_cast<double*>(cst) + s, Sc}, lc, C::NSEG);
  for (int e = 0; e < C::n; ++e) la(e) = 0.0;
  for (int t = t0; t < t1; ++t) {
    const int st = (t - t0) % PAR_NST;
    const double* stg = ring.wait(st);
    WView lv = ring.view(stg, 0), kv = ring.view(stg, 2 * DM::EL), cvw = ring.view(stg, 2 * (DM::EL + DM::EK));
    FView sfv = ring.fview(stg, 2 * (DM::EL + DM::EK + DM::EC)), sgv = ring.fview(stg, 2 * (DM::EL + DM::EK + DM::EC) + SR::NSF);
    const float* fr = ring.frow(stg);
    double Cm[R * R], Lt[U * B], Kt[B * Y];
    LQGK_UNROLL for (int i = 0; i < U * B; ++i) Lt[i] = lv(i);
    LQGK_UNROLL for (int i = 0; i < B * Y; ++i) Kt[i] = kv(i);
    load_sym_ws<R>(cvw, 0, Cm);
    auto sf = [&](int e) { return sfv(e); };
    auto get = [&](int idx) { return fr[idx]; };
    auto out = [&](int e, double v) { la(e) += v; };
    double Kb[B * Y];
    if constexpr (P0) {
      double Lb[U * B];
      CC::pass0(lc, [&](int e) { return sgv(e); }, t == 0, [&](int e) { return SGBI[(size_t)e * Sc + s]; }, sf, get, Cm, Lt, Kt, out,
                Lb, Kb);
      LQGK_UNROLL for (int i = 0; i < U * B; ++i) Lbar[((size_t)t * DM::EL + i) * Sc + s] = Lb[i];
      if constexpr (!P1) { LQGK_UNROLL for (int i = 0; i < B * Y; ++i) Kbar[((size_t)t * DM::EK + i) * Sc + s] = Kb[i]; }
    } else {
      LQGK_UNROLL for (int i = 0; i < B * Y; ++i) Kb[i] = 0.0;
    }
    if constexpr (P1) {
      CC::pass1(lc, sf, get, Cm, Lt, Kt, out, Kb);
      // PASS 1 alone stores the transition part separately (k_kf_rev adds the two parts); PASS 2 stores the total
      double* dst = PASS == 1 ? KbarF : Kbar;
      LQGK_UNROLL for (int i = 0; i < B * Y; ++i) dst[((size_t)t * DM::EK + i) * Sc + s] = Kb[i];
      if constexpr (PASS == 2) { LQGK_UNROLL for (int i = 0; i < B * Y; ++i) KbarF[((size_t)t * DM::EK + i) * Sc + s] = 0.0; }
    }
    __syncwarp();
    if (t + PAR_NST < t1) ring.issue(t + PAR_NST, st);
  }
  flush_acc_atomic<C>(acc + s, Sc, la, C::NSEG);
}

// Kalman-gain adjoint (sequential, t descending).  Ring inputs per step: P_t, Kbar_t.
// [t0, t1) walked downwards; `carry` ([B*B][Sc]) hands the cotangent of P from one launch to the next (see k_cov_seq_rev).
template <class DM>
__global__ void __launch_bounds__(32) k_kf_rev(const double* cst, size_t Sc, int Tn, const double* Pkf, const double* Kbar,
                                               const double* KbarF, double* acc, int t0, int t1, double* carry) {
  extern __shared__ __align__(128) double sm[];
  constexpr int B = DM::B, Y = DM::Y;
  using C = KfC<DM>;
  using Ring = StepRing<3, SEQ_NST>;
  constexpr int ROWS = DM::EP + 2 * DM::EK;
  const int lane = threadIdx.x;
  const size_t s0 = (size_t)blockIdx.x * 32, s = s0 + lane;
  double* lcp = sm + (size_t)SEQ_NST * ROWS * 32;
  double* lap = lcp + C::n * 32;
  uint64_t* bars = reinterpret_cast<uint64_t*>(lap + C::n * 32);
  Ring ring{{{Pkf + s0, DM::EP, 0}, {Kbar + s0, DM::EK, 0}, {KbarF + s0, DM::EK, 0}}, Sc, nullptr, 0, 0, 0, sm, bars, lane, 2 * ROWS, ROWS * 32, 0};
  ring.init();
  const int nsteps = t1 - t0;
  for (int k = 0; k < SEQ_NST && k < nsteps; ++k) ring.issue(t1 - 1 - k, k);
  WView lc{lcp + lane, 32}, la{lap + lane, 32};
  load_consts<C>(WView{const_cast<double*>(cst) + s, Sc}, lc, C::NSEG);
  for (int e = 0; e < C::n; ++e) la(e) = 0.0;
  auto accf = [&](int e) -> double& { return la(e); };
  double Pnb[B * B];
  if (t1 == Tn) { LQGK_UNROLL for (int i = 0; i < B * B; ++i) Pnb[i] = 0.0; }
  else { LQGK_UNROLL for (int i = 0; i < B * B; ++i) Pnb[i] = carry[(size_t)i * Sc + s]; }
  auto sweep = [&](const auto& cv) {
    for (int kk = 0; kk < nsteps; ++kk) {
      const int st = kk % SEQ_NST;
      const double* stg = ring.wait(st);
      double P[B * B], Kb[B * Y];
      load_sym_ws<B>(ring.view(stg, 0), 0, P);
      {
        WView kv = ring.view(stg, 2 * DM::EP), kv2 = ring.view(stg, 2 * (DM::EP + DM::EK));
        LQGK_UNROLL for (int i = 0; i < B * Y; ++i) Kb[i] = kv(i) + kv2(i);
      }
      __syncwarp();
      if (kk + SEQ_NST < nsteps) ring.issue(t1 - 1 - (kk + SEQ_NST), st);
      KfRev<DM>::step(cv, accf, P, Kb, Pnb);
    }
  };
  if constexpr (C::n <= LQGK_REG_CONSTS_MAX) {
    RegView<C::n> rc;
    LQGK_UNROLL for (int e = 0; e < C::n; ++e) rc.v[e] = lc(e);
    sweep(rc);
  } else {
    sweep(lc);
  }
  if (t0 == 0) KfRev<DM>::finish(accf, Pnb);
  else { LQGK_UNROLL for (int i = 0; i < B * B; ++i) carry[(size_t)i * Sc + s] = Pnb[i]; }
  flush_acc_atomic<C>(acc + s, Sc, la, C::NSEG);
}

// Riccati adjoint (sequential, t ascending).  Ring inputs per step: S_{t+1}, L_t, Lbar_t.
template <class DM>
__global__ void __launch_bounds__(32) k_lqr_rev(const double* cst, size_t Sc, int Tn, double eps, const double* L,
                                                const double* Sric, const double* Lbar, double* acc) {
  extern __shared__ __align__(128) double sm[];
  constexpr int B = DM::B, U = DM::U;
  using C = LqrC<DM>;
  using Ring = StepRing<3, SEQ_NST>;
  constexpr int ROWS = DM::ES + 2 * DM::EL;
  const int lane = threadIdx.x;
  const size_t s0 = (size_t)blockIdx.x * 32, s = s0 + lane;
  double* lcp = sm + (size_t)SEQ_NST * ROWS * 32;
  double* lap = lcp + C::n * 32;
  uint64_t* bars = reinterpret_cast<uint64_t*>(lap + C::n * 32);
  Ring ring{{{Sric + s0, DM::ES, 0}, {L + s0, DM::EL, 0}, {Lbar + s0, DM::EL, 0}}, Sc, nullptr, 0, 0, 0, sm, bars, lane, 2 * ROWS, ROWS * 32, 0};
  ring.init();
  for (int k = 0; k < SEQ_NST && k < Tn; ++k) ring.issue(k, k);
  WView lc{lcp + lane, 32}, la{lap + lane, 32};
  load_consts<C>(WView{const_cast<double*>(cst) + s, Sc}, lc, C::NSEG);
  for (int e = 0; e < C::n; ++e) la(e) = 0.0;
  auto accf = [&](int e) -> double& { return la(e); };
  double Sn[B * B];
  LQGK_UNROLL for (int i = 0; i < B * B; ++i) Sn[i] = 0.0;
  auto sweep = [&](const auto& cv) {
    for (int t = 0; t < Tn; ++t) {
      const int st = t % SEQ_NST;
      const double* stg = ring.wait(st);
      double S[B * B], Lt[U * B], Lb[U * B];
      load_sym_ws<B>(ring.view(stg, 0), 0, S);
      {
        WView lv = ring.view(stg, 2 * DM::ES), bv = ring.view(stg, 2 * (DM::ES + DM::EL));
        LQGK_UNROLL for (int i = 0; i < U * B; ++i) { Lt[i] = lv(i); Lb[i] = bv(i); }
      }
      __syncwarp();
      if (t + SEQ_NST < Tn) ring.issue(t + SEQ_NST, st);
      double shift;
      {
        double Bm[B * U], SB[B * U], H[U * U];
        load_mat<B, U>(cv, C::Ba, Bm);
        mm<B, B, U>(S, Bm, SB);
        load_sym<U>(cv, C::R, H);
        mm_tn_sym<U, B, true>(Bm, SB, H);
        shift = eps - lambda_min<U>(H);
        shift = shift > 0.0 ? shift : 0.0;
      }
      LqrRev<DM>::step(cv, accf, S, Lt, Lb, shift, Sn);
    }
  };
  if constexpr (C::n <= LQGK_REG_CONSTS_MAX) {
    RegView<C::n> rc;
    LQGK_UNROLL for (int e = 0; e < C::n; ++e) rc.v[e] = lc(e);
    sweep(rc);
  } else {
    sweep(lc);
  }
  LqrRev<DM>::finish(accf, Sn);
  flush_acc_atomic<C>(acc + s, Sc, la, C::NSEG);
}

// Dynamic shared-memory sizes of the per-sample kernels (must mirror the carve-up inside each kernel).
template <class DM> constexpr size_t smem_cov_fwd() {
  return sizeof(double) * ((size_t)SEQ_NST * (DM::EL + DM::EK) * 32 + CovC<DM>::n * 32) +
         sizeof(float) * SmemRecSink<DM>::FLOATS + sizeof(uint64_t) * SEQ_NST;
}
template <class DM> constexpr size_t smem_cov_seq_rev() {
  using SR = CovSeqRev<DM>;
  return sizeof(double) * ((size_t)SEQ_NST * StepRing<2, SEQ_NST>::stage_size(SR::NSF + SR::NJS, DM::SUMP - DM::SUM_J) + SR::SC_N * 32) +   // float rows
         sizeof(uint64_t) * SEQ_NST;
}
template <class DM, int PASS> constexpr size_t smem_cov_contrib() {
  using SR = CovSeqRev<DM>;
  constexpr int UNITS = 2 * (DM::EL + DM::EK + DM::EC) + SR::NSF + (PASS != 1 ? SR::NSGB : 0);
  constexpr int PAR_NST = contrib_nst<DM, PASS>();
  return sizeof(double) * ((size_t)PAR_NST * StepRing<5, PAR_NST>::stage_size(UNITS, DM::SUM_J) + 2 * CovC<DM>::n * 32) +
         sizeof(uint64_t) * PAR_NST;
}
template <class DM> constexpr size_t smem_kf_rev() {
  return sizeof(double) * ((size_t)SEQ_NST * (DM::EP + 2 * DM::EK) * 32 + 2 * KfC<DM>::n * 32) + sizeof(uint64_t) * SEQ_NST;
}
template <class DM> constexpr size_t smem_lqr_rev() {
  return sizeof(double) * ((size_t)SEQ_NST * (DM::ES + 2 * DM::EL) * 32 + 2 * LqrC<DM>::n * 32) + sizeof(uint64_t) * SEQ_NST;
}

// =========================================================================================== per-trial kernels
// Resident CTAs per SM the forward per-trial kernel is compiled for: the small systems are latency-bound at 2 CTAs (8 warps)
// per SM, so the register budget is capped at 65536 / (3 * 128) = 170 to fit 3.
// The adjoint kernel needs ~240 registers; capped at 170 it spills and runs 1.6x slower (measured), so it stays at 2 CTAs.
#ifndef LQGK_FWD_WARPS
#define LQGK_FWD_WARPS 4
#endif
constexpr int TRIAL_WARPS = LQGK_FWD_WARPS;   // warps (= samples) per CTA of the forward kernel
template <class DM>
__host__ __device__ constexpr int trial_min_ctas() { return DM::N <= 6 ? 12 / TRIAL_WARPS : 1; }
#ifndef LQGK_REV_WARPS
#define LQGK_REV_WARPS 4
#endif
constexpr int TRIAL_WARPS_REV = LQGK_REV_WARPS;   // ... and of the adjoint kernel
// time steps per ring stage of the forward kernel: 8 for the small records, fewer when one record is KBs (large systems)
template <class DM>
__host__ __device__ constexpr int trial_tb() { return DM::REC <= 128 ? 8 : (DM::REC <= 256 ? 4 : 2); }
constexpr int TRIAL_NST = 3;     // ring stages of the forward kernel

constexpr int TRIAL_PF = 4;      // observation prefetch distance in time steps (cp.async groups in flight)
// Sums over trials in the adjoint: every lane holds 32 partial values; they are transposed through shared memory (lane L
// writes its 32 values as 8 x 128-bit stores into row L of a [32][36] tile -- conflict-free per quarter warp --, then sums
// column L: 32 conflict-free loads) instead of a 31-shuffle butterfly with 62 selects.
constexpr int TRIAL_RED_STRIDE = 36;

// ------------------------------------------------------------------------------------------- checkpointed state history
// The adjoint needs the carried mean c_t of every trial at every step.  The forward kernel stores c_t only at the segment
// starts t = k * CK ("checkpoints"); the adjoint kernel processes one segment at a time: it re-runs the state recursion from
// the checkpoint (Trial::advance, CK - 1 steps, bit-identical to the forward pass) into a per-warp shared-memory buffer
// [CK][R][32 RT] and then walks the segment backwards reading c_t from that buffer.  CK = 1 stores every step (no
// recomputation).  CK is bounded by the per-warp share of shared memory that keeps 2 CTAs (8 warps) resident per SM.
#ifndef LQGK_TRIAL_CK_MAX
#define LQGK_TRIAL_CK_MAX 8
#endif
constexpr int TRIAL_CK_MAX = LQGK_TRIAL_CK_MAX;
#ifndef LQGK_TRIAL_WARP_SMEM
#define LQGK_TRIAL_WARP_SMEM 28440    // bytes per warp: 2 CTAs x 4 warps x 28,440 B + 2 KB reserved < 228 KB per SM
#endif
template <class DM>
__host__ __device__ constexpr int trial_red_bytes() { return DM::NSUM >= 32 ? 32 * TRIAL_RED_STRIDE * (int)sizeof(float) : 0; }
template <class DM>
__host__ __device__ constexpr int trial_ck(int RT) {
  const int per_step = 2 * DM::REC * (int)sizeof(float) + DM::R * 32 * RT * (int)sizeof(float);   // 2 ring stages + 1 state slot
  const int ck = (LQGK_TRIAL_WARP_SMEM - trial_red_bytes<DM>() - 16) / per_step;
  return ck < 1 ? 1 : (ck > TRIAL_CK_MAX ? TRIAL_CK_MAX : ck);
}
// Largest number of trials one lane carries: small systems leave room for 8 (amortises the broadcast record loads and
// the cross-lane reductions over more FMAs), large ones for 4.
template <class DM>
__host__ __device__ constexpr int trial_rt_max() { return DM::N * DM::N <= 36 ? 8 : 4; }
__host__ __device__ __forceinline__ constexpr int trial_rt(int N, int rt_max) { return (N + 31) / 32 < rt_max ? (N + 31) / 32 : rt_max; }
// Geometry of the per-trial kernels for N trials: RT trials per lane, NB passes ("blocks") of ROW = 32 RT trials, CK steps per
// segment.  Checkpoints are laid out [s][segment][NB][R][ROW], repacked observations [(s)][T+1][NB][D][ROW] (k_repack_obs).
struct TrialGeom {
  int RT, ROW, NB, CK, nseg;
};
template <class DM>
__host__ __device__ constexpr TrialGeom trial_geom(int N, int T) {
  const int rt = trial_rt(N, trial_rt_max<DM>());
  const int ck = trial_ck<DM>(rt);
  return TrialGeom{rt, 32 * rt, (N + 32 * rt - 1) / (32 * rt), ck, (T + ck - 1) / ck};
}

template <class DM, int RT, bool REV>
constexpr size_t trial_smem_bytes() {
  if constexpr (REV) {
    constexpr int CK = trial_ck<DM>(RT);
    return (size_t)TRIAL_WARPS_REV * (2 * CK * DM::REC * sizeof(float) + 2 * sizeof(uint64_t) + trial_red_bytes<DM>() +
                                  (size_t)CK * DM::R * 32 * RT * sizeof(float));
  } else {
    size_t ring = (size_t)TRIAL_WARPS * TRIAL_NST * trial_tb<DM>() * DM::REC * sizeof(float) + TRIAL_WARPS * TRIAL_NST * sizeof(uint64_t);
    size_t pf = (size_t)TRIAL_WARPS * (TRIAL_PF + 1) * RT * 32 * DM::D * sizeof(float);
    return ring + pf;
  }
}

// Per-warp ring of NST record chunks of TB time steps, filled by bulk async copies.  Chunk k covers steps
// [k*TB, min(T,(k+1)*TB)).
template <class DM, int TB, int NST>
struct RecRing {
  float* buf;        // [NST][TB*REC]
  uint64_t* bars;    // [NST]
  const float* src;  // this sample's records [Tn][REC]
  int Tn, lane;
  uint32_t phase_bits;
  __device__ __forceinline__ void init() {
    if (lane == 0) {
      for (int i = 0; i < NST; ++i) mbar_init(&bars[i], 1);
      fence_mbar_init();
    }
    phase_bits = 0;
    __syncwarp();
  }
  // issue the copy of chunk `k` into stage `st` (lane 0 only; caller guarantees the stage is no longer read)
  __device__ __forceinline__ void issue(int k, int st) {
    if (lane == 0) {
      int t0 = k * TB;
      int nst = min(TB, Tn - t0);
      uint32_t bytes = (uint32_t)nst * DM::REC * sizeof(float);
      fence_proxy_async();
      mbar_expect_tx(&bars[st], bytes);
      bulk_g2s(buf + (size_t)st * TB * DM::REC, src + (size_t)t0 * DM::REC, bytes, &bars[st]);
    }
  }
  __device__ __forceinline__ const float* wait(int st) {
    mbar_wait(&bars[st], (phase_bits >> st) & 1u);
    phase_bits ^= (1u << st);
    return buf + (size_t)st * TB * DM::REC;
  }
};

// Trial -> lane assignment inside one block of ROW = 32 RT trials: pair p of a lane holds the ADJACENT trials (columns)
// 64p + 2*lane and +1, so one 64-bit access moves the pair's entry of a checkpoint or of an observation row, already in f32x2
// register order (no packing moves, half the memory instructions); an odd RT adds the single column 64*(RT/2) + lane.
// Flat slot j: 2p, 2p+1 = the two halves of pair p; RT-1 = the single.
template <int RT>
__device__ __forceinline__ int trial_col(int lane, int j) {
  constexpr int NP = RT / 2;
  return j < 2 * NP ? 64 * (j >> 1) + 2 * lane + (j & 1) : 64 * NP + lane;
}
// A lane's view of one row block [M][ROW] (a checkpoint, a shared-memory state slot or an observation row; M components)
// through two pointers: pp = block + 2 lane (pair p, component m at pp[m ROW + 64 p], 64 bits), ps = block + 64 NP + lane
// (the single at ps[m ROW]).  Every offset is a compile-time immediate.
template <int RT, int M>
struct LaneBlock {
  static constexpr int NP = RT / 2, NS = RT % 2, NPA = NP > 0 ? NP : 1, ROW = 32 * RT;
  template <bool LDG>
  __device__ __forceinline__ static void load(const float* pp, const float* ps, f32x2 (&vp)[NPA][M], float (&vs)[M]) {
    LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) LQGK_UNROLL for (int m = 0; m < M; ++m) {
      const float2* a = reinterpret_cast<const float2*>(pp + m * ROW + 64 * p2);
      float2 v = LDG ? __ldg(a) : *a;
      vp[p2][m] = f32x2{v.x, v.y};
    }
    if constexpr (NS) { LQGK_UNROLL for (int m = 0; m < M; ++m) vs[m] = LDG ? __ldg(ps + m * ROW) : ps[m * ROW]; }
  }
  __device__ __forceinline__ static void store(float* pp, float* ps, const f32x2 (&vp)[NPA][M], const float (&vs)[M]) {
    LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) LQGK_UNROLL for (int m = 0; m < M; ++m)
      *reinterpret_cast<float2*>(pp + m * ROW + 64 * p2) = make_float2(vp[p2][m].x, vp[p2][m].y);
    if constexpr (NS) { LQGK_UNROLL for (int m = 0; m < M; ++m) ps[m * ROW] = vs[m]; }
  }
  __device__ __forceinline__ static void store_streaming(float* pp, float* ps, const f32x2 (&vp)[NPA][M], const float (&vs)[M]) {
    LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) LQGK_UNROLL for (int m = 0; m < M; ++m)
      __stcs(reinterpret_cast<float2*>(pp + m * ROW + 64 * p2), make_float2(vp[p2][m].x, vp[p2][m].y));   // written once, read once
    if constexpr (NS) { LQGK_UNROLL for (int m = 0; m < M; ++m) __stcs(ps + m * ROW, vs[m]); }
  }
  // global -> shared, asynchronously (LDGSTS); dp/ds: this lane's pointers into the shared-memory block
  __device__ __forceinline__ static void copy_async(float* dp, float* ds, const float* pp, const float* ps) {
    LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) LQGK_UNROLL for (int m = 0; m < M; ++m)
      cp_async<8>(dp + m * ROW + 64 * p2, pp + m * ROW + 64 * p2);
    if constexpr (NS) { LQGK_UNROLL for (int m = 0; m < M; ++m) cp_async<4>(ds + m * ROW, ps + m * ROW); }
    cp_async_commit();
  }
};

// Copy one step's record from the shared-memory ring into registers (small systems) with 128-bit broadcast loads.
template <class DM>
struct RecRegs {
  float v[DM::REC];
  __device__ __forceinline__ void load(const float* r) {
    const float4* r4 = reinterpret_cast<const float4*>(r);
    LQGK_UNROLL for (int k = 0; k < DM::REC / 4; ++k) {
      float4 q = r4[k];
      v[4 * k] = q.x; v[4 * k + 1] = q.y; v[4 * k + 2] = q.z; v[4 * k + 3] = q.w;
    }
  }
  __device__ __forceinline__ float operator[](int i) const { return v[i]; }
};
template <class DM>
__host__ __device__ constexpr bool rec_in_regs() { return DM::REC <= 48; }

// Forward: per-trial mean recursion + log-density.  grid = (ceil(n_samples / TRIAL_WARPS)), block = 32 * TRIAL_WARPS.
// Trials are processed in NB passes of ROW = 32*RT.  Observations (blocked component-major, k_repack_obs) are prefetched
// TRIAL_PF steps ahead with per-lane cp.async copies into shared-memory slots laid out like the source block ([D][ROW]: no
// registers held, no stalls on the L2 round trip) and read back as f32x2 pairs.
// `hist` (VJP only): checkpoints of the carried state at the segment starts, [s][segment][NB][R][ROW].
template <class DM, int RT>
__global__ void __launch_bounds__(32 * TRIAL_WARPS, trial_min_ctas<DM>()) k_trial_fwd(const float* __restrict__ rec, const float* __restrict__ xc_all,
                                                                size_t xc_sample_stride, int n_samples, int N, int Tn,
                                                                double* __restrict__ ll_ws, float* __restrict__ hist, int ka, int kb) {
  // [ka, kb): range of checkpoint segments (CK steps each) of this launch.  ka > 0 continues from checkpoint ka (needs `hist`)
  // and adds its log-density terms to what the earlier launches left in ll_ws (pipelined launch sequence).
  constexpr int D = DM::D, R = DM::R, NSLOT = TRIAL_PF + 1, TB = trial_tb<DM>(), CK = trial_ck<DM>(RT), ROW = 32 * RT;
  constexpr int NP = RT / 2, NS = RT % 2, NPA = NP > 0 ? NP : 1;
  using XB = LaneBlock<RT, D>;
  using CB = LaneBlock<RT, R>;
  extern __shared__ __align__(128) unsigned char smraw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int s = blockIdx.x * TRIAL_WARPS + warp;
  if (s >= n_samples) return;
  const int NB = (N + ROW - 1) / ROW;
  const float* __restrict__ xc = xc_all + (size_t)s * xc_sample_stride;   // this sample's observations [T+1][NB][D][ROW]
  constexpr size_t RING_BYTES = (size_t)TRIAL_WARPS * TRIAL_NST * TB * DM::REC * sizeof(float);
  float* ring_base = reinterpret_cast<float*>(smraw);
  uint64_t* bar_base = reinterpret_cast<uint64_t*>(smraw + RING_BYTES);
  float* pf = reinterpret_cast<float*>(smraw + RING_BYTES + TRIAL_WARPS * TRIAL_NST * sizeof(uint64_t)) + (size_t)warp * NSLOT * D * ROW;
  const int ta = ka * CK, tb = min(Tn, kb * CK), Tl = tb - ta;     // time range of this launch
  RecRing<DM, TB, TRIAL_NST> ring{ring_base + (size_t)warp * TRIAL_NST * TB * DM::REC, bar_base + warp * TRIAL_NST,
                                  rec + ((size_t)s * Tn + ta) * DM::REC, Tl, lane, 0};   // ring chunks relative to ta
  ring.init();
  const int nchunk = (Tl + TB - 1) / TB;
  const int nseg = (Tn + CK - 1) / CK;
  const size_t xstep = (size_t)NB * D * ROW, hstep = (size_t)NB * R * ROW;
  const int lp = 2 * lane, ls = 64 * NP + lane;                       // this lane's pair / single column inside a block
  for (int blk = 0; blk < NB; ++blk) {
    const float* xlp = xc + (size_t)blk * D * ROW + lp + (size_t)ta * xstep;   // row ta of this block; row t at + (t - ta) * xstep
    const float* xls = xc + (size_t)blk * D * ROW + ls + (size_t)ta * xstep;
    float* hp = hist + (((size_t)s * nseg + ka) * NB + blk) * R * ROW + lp;   // checkpoint ka; advanced by hstep per stored checkpoint
    float* hs = hist + (((size_t)s * nseg + ka) * NB + blk) * R * ROW + ls;
    int ckc = 0;                     // steps until the next checkpoint
    // trials 2p, 2p+1 are packed into one f32x2 lane-pair state (Blackwell FFMA2); an odd last trial stays scalar
    f32x2 cP[NPA][R], x0P[NPA][D];
    float cS[R], x0S[D];
    double ll[RT];
    LQGK_UNROLL for (int j = 0; j < RT; ++j) ll[j] = 0.0;
    XB::template load<true>(xlp, xls, x0P, x0S);
    if (ka == 0) {
      LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) LQGK_UNROLL for (int k = 0; k < R; ++k) cP[p2][k] = f32x2{0.f, 0.f};
      LQGK_UNROLL for (int k = 0; k < R; ++k) cS[k] = 0.f;
    } else {
      CB::template load<true>(hp, hs, cP, cS);   // c_{ta} as the previous launch stored it
    }
    // prologue: x_{ta+1..ta+PF} in flight (one commit group per step); xnp/xns walk one row per step, clamped at row Tn
    const float* xnp = xlp;
    const float* xns = xls;
    int trow = ta;                   // row xnp/xns point at
    auto advance_row = [&]() { if (trow < Tn) { ++trow; xnp += xstep; xns += xstep; } };
    for (int p = 0; p < TRIAL_PF; ++p) {
      advance_row();
      float* slot = pf + (p % NSLOT) * (D * ROW);
      XB::copy_async(slot + lp, slot + ls, xnp, xns);
    }
    for (int k = 0; k < TRIAL_NST && k < nchunk; ++k) ring.issue(k, k);
    int wslot = TRIAL_PF % NSLOT, rslot = 0;       // prefetch slot being filled / slot holding x_{t+1}
    for (int k = 0; k < nchunk; ++k) {
      const int st = k % TRIAL_NST;
      const float* chunk = ring.wait(st);
      const int t0 = k * TB, nst = min(TB, Tl - t0);
      f32x2 partP[NPA];
      float partS = 0.f;
      LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) partP[p2] = f32x2{0.f, 0.f};
#pragma unroll 1
      for (int q = 0; q < nst; ++q) {
        const float* r = chunk + q * DM::REC;
        f32x2 x1P[NPA][D];
        float x1S[D];
        {   // prefetch x_{t+1+PF}, then make sure x_{t+1} has landed
          advance_row();
          float* slot = pf + wslot * (D * ROW);
          XB::copy_async(slot + lp, slot + ls, xnp, xns);
          cp_async_wait<TRIAL_PF>();
          const float* cur = pf + rslot * (D * ROW);
          XB::template load<false>(cur + lp, cur + ls, x1P, x1S);
          wslot = wslot + 1 == NSLOT ? 0 : wslot + 1;
          rslot = rslot + 1 == NSLOT ? 0 : rslot + 1;
        }
        if (hist != nullptr) {
          if (ckc == 0) {            // t is a segment start: store the checkpoint c_t
            ckc = CK;
            CB::store_streaming(hp, hs, cP, cS);
            hp += hstep;
            hs += hstep;
          }
          --ckc;
        }
        auto run = [&](const auto& rr) {
          LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2)
            partP[p2] = Ops<f32x2>::add(partP[p2], Trial<DM>::template fwd<f32x2>(rr, x0P[p2], x1P[p2], cP[p2]));
          if constexpr (NS) partS += Trial<DM>::template fwd<float>(rr, x0S, x1S, cS);
        };
        if constexpr (rec_in_regs<DM>()) {
          RecRegs<DM> rr;
          rr.load(r);
          run(rr);
        } else {
          run(r);
        }
        LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) LQGK_UNROLL for (int m = 0; m < D; ++m) x0P[p2][m] = x1P[p2][m];
        if constexpr (NS) { LQGK_UNROLL for (int m = 0; m < D; ++m) x0S[m] = x1S[m]; }
      }
      // FP32 partial sum over <= TB steps, FP64 across chunks (log-likelihood error ~1e-7 relative)
      LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) {
        ll[2 * p2] += (double)partP[p2].x;
        ll[2 * p2 + 1] += (double)partP[p2].y;
      }
      if constexpr (NS) ll[RT - 1] += (double)partS;
      __syncwarp();
      if (k + TRIAL_NST < nchunk) ring.issue(k + TRIAL_NST, st);
    }
    cp_async_wait<0>();
    if (hist != nullptr && kb < nseg) CB::store_streaming(hp, hs, cP, cS);   // checkpoint kb: where the next launch continues from
    LQGK_UNROLL for (int j = 0; j < RT; ++j) {
      const int i = blk * ROW + trial_col<RT>(lane, j);
      if (i < N) {
        if (ka == 0) ll_ws[(size_t)s * N + i] = ll[j];
        else ll_ws[(size_t)s * N + i] += ll[j];
      }
    }
  }
}

// Transposing butterfly over V = 2^k <= 32 values: every lane holds V partial values; afterwards the lanes whose top
// log2(V) lane-index bits equal i hold the warp-wide total of value i (V == 32: lane L holds value L).
template <int V>
__device__ __forceinline__ float warp_transpose_reduce(float (&val)[V], int lane) {
  int bit = 16;
  LQGK_UNROLL for (int h = V / 2; h >= 1; h >>= 1) {
    const bool up = (lane & bit) != 0;
    LQGK_UNROLL for (int j = 0; j < h; ++j) {
      float send = up ? val[j] : val[j + h];
      float keep = up ? val[j + h] : val[j];
      val[j] = keep + __shfl_xor_sync(FULL, send, bit);
    }
    bit >>= 1;
  }
  float tot = val[0];
  LQGK_UNROLL for (int m = 16 / V; m >= 1; m >>= 1) tot += __shfl_xor_sync(FULL, tot, m);
  return tot;
}
__host__ __device__ constexpr int pow2_ceil(int v) { return v <= 1 ? 1 : (v <= 2 ? 2 : (v <= 4 ? 4 : (v <= 8 ? 8 : (v <= 16 ? 16 : 32)))); }

// Reverse: per-trial adjoint, segment by segment from the last one: (1) the checkpoint c_{k CK} arrives in the segment
// buffer by per-lane cp.async (issued one segment ahead into the slot the previous segment freed first), (2) the state
// recursion is re-run forward through the segment, c_t -> buffer slot t - k CK, (3) the adjoint walks the segment backwards
// reading c_t from the buffer, and writes the per-step sums over trials (DM::SUM_* layout) to sums[s][t][SUMP].  Every buffer
// entry is private to the lane that owns the trial, so no warp synchronisation is needed around it.  Passes over trial blocks
// accumulate (+=) into the sums.
//
// The backward walk is written as two alternating copies of the step (ping-pong): the cotangent cb and the observation rows
// live in two register sets that swap roles every step, so nothing is copied from "next" to "current" at the loop edge
// (those copies and the pairing of trial-major observations were a quarter of the instructions of the first version).
#ifndef LQGK_REV_MIN_CTAS
#define LQGK_REV_MIN_CTAS 1
#endif
#ifndef LQGK_REV_REC_REGS
#define LQGK_REV_REC_REGS 1
#endif
template <class DM, int RT>
#if LQGK_REV_MIN_CTAS > 1
__global__ void __launch_bounds__(32 * TRIAL_WARPS_REV, LQGK_REV_MIN_CTAS) k_trial_rev(
#else
__global__ void __launch_bounds__(32 * TRIAL_WARPS_REV) k_trial_rev(
#endif
    const float* __restrict__ rec, const float* __restrict__ xc_all,
                                                                size_t xc_sample_stride, const float* __restrict__ hist,
                                                                const float* __restrict__ w, int n_samples, int N, int Tn,
                                                                float* __restrict__ sums, int ka, int kb, float* __restrict__ cbcar) {
  // [ka, kb): range of checkpoint segments of this launch, walked downwards.  kb < nseg starts from the cotangent an earlier
  // launch left in cbcar ([s][NB][R][ROW]); ka > 0 leaves its own there (pipelined launch sequence).
  constexpr int D = DM::D, R = DM::R;
  constexpr int CK = trial_ck<DM>(RT), ROW = 32 * RT, SLOT = R * ROW;
  constexpr int NFULL = DM::NSUM / 32, REM = DM::NSUM % 32, VREM = pow2_ceil(REM);
  constexpr int NP = RT / 2, NS = RT % 2, NPA = NP > 0 ? NP : 1;
  using XB = LaneBlock<RT, D>;
  using CB = LaneBlock<RT, R>;
  extern __shared__ __align__(128) unsigned char smraw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int s = blockIdx.x * TRIAL_WARPS_REV + warp;
  if (s >= n_samples) return;
  const int NB = (N + ROW - 1) / ROW;
  const float* __restrict__ xc = xc_all + (size_t)s * xc_sample_stride;   // this sample's observations [T+1][NB][D][ROW]
  constexpr size_t RING_FLOATS = (size_t)2 * CK * DM::REC;
  float* ring_base = reinterpret_cast<float*>(smraw);
  uint64_t* bar_base = reinterpret_cast<uint64_t*>(ring_base + TRIAL_WARPS_REV * RING_FLOATS);
  float* red_base = reinterpret_cast<float*>(bar_base + TRIAL_WARPS_REV * 2);                     // 16-byte aligned
  float* red = red_base + (size_t)warp * (trial_red_bytes<DM>() / sizeof(float));
  float* seg = red_base + (size_t)TRIAL_WARPS_REV * (trial_red_bytes<DM>() / sizeof(float)) + (size_t)warp * CK * SLOT;
  RecRing<DM, CK, 2> ring{ring_base + (size_t)warp * RING_FLOATS, bar_base + warp * 2, rec + (size_t)s * Tn * DM::REC, Tn, lane, 0};
  ring.init();
  const int nseg = (Tn + CK - 1) / CK;
  const size_t xstep = (size_t)NB * D * ROW, hstep = (size_t)NB * R * ROW;
  const int lp = 2 * lane, ls = 64 * NP + lane;                       // this lane's pair / single column inside a block
  for (int blk = 0; blk < NB; ++blk) {
    float wt[RT];
    LQGK_UNROLL for (int j = 0; j < RT; ++j) {
      const int i = blk * ROW + trial_col<RT>(lane, j);
      wt[j] = i < N ? w[(size_t)s * N + i] : 0.f;  // columns beyond the last trial: w = 0, cb stays 0, their data are finite
    }
    const float* xlp = xc + (size_t)blk * D * ROW + lp;              // row 0 of this block; row t at + t * xstep
    const float* xls = xc + (size_t)blk * D * ROW + ls;
    auto next_slot = [&](float* p) { p += SLOT; return p == seg + CK * SLOT ? seg : p; };
    auto prev_slot = [&](float* p) { return (p == seg ? seg + CK * SLOT : p) - SLOT; };
    // Ping-pong state of the backward walk.  A step of parity P reads the cotangent from cb[P] and leaves the next one in
    // cb[P ^ 1]; it takes x_t from x[P] and x_{t+1} from x[P ^ 1] (the previous step's x_t) and, once the residual no longer
    // needs x_{t+1}, requests x_{t-1} into x[P ^ 1].  A segment's walk starts with parity 1; after an even number of steps the
    // carried state sits again where the next walk expects it (cb[1], x_{t+1} in x[0]).
    f32x2 cbP[2][NPA][R], xP[2][NPA][D], wP[NPA];
    float cbS[2][R], xS[2][D], wS = wt[RT - 1];
    const int tend = min(Tn, kb * CK);             // one past the last step of this launch
    XB::template load<true>(xlp + (size_t)tend * xstep, xls + (size_t)tend * xstep, xP[0], xS[0]);
    LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) wP[p2] = f32x2{wt[2 * p2], wt[2 * p2 + 1]};
    float* carp = cbcar + ((size_t)s * NB + blk) * R * ROW + lp;
    float* cars = cbcar + ((size_t)s * NB + blk) * R * ROW + ls;
    if (kb == nseg) {
      LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) LQGK_UNROLL for (int k = 0; k < R; ++k) cbP[1][p2][k] = f32x2{0.f, 0.f};
      LQGK_UNROLL for (int k = 0; k < R; ++k) cbS[1][k] = 0.f;
    } else {
      CB::template load<true>(carp, cars, cbP[1], cbS[1]);
    }
    const float* hkp = hist + (((size_t)s * nseg + (kb - 1)) * NB + blk) * R * ROW + lp;   // checkpoint of the segment to fetch next
    const float* hks = hist + (((size_t)s * nseg + (kb - 1)) * NB + blk) * R * ROW + ls;
    float* slot0 = seg;                            // buffer slot of the current segment's first step
    CB::copy_async(slot0 + lp, slot0 + ls, hkp, hks);
    ring.issue(kb - 1, 0);
    if (kb - ka > 1) ring.issue(kb - 2, 1);
    float* out = sums + ((size_t)s * Tn + (tend - 1)) * DM::SUMP;
    const int nloc = kb - ka;
    for (int kk = 0; kk < nloc; ++kk) {
      const int k = kb - 1 - kk, st = kk & 1;
      const int t0 = k * CK, nst = min(CK, Tn - t0);
      const float* chunk = ring.wait(st);
      cp_async_wait<0>();                          // checkpoint k is in slot0 (lane-private data: no warp sync needed)
      const float* xsp = xlp + (size_t)t0 * xstep;  // observation row t0 of this lane (pairs / single)
      const float* xss = xls + (size_t)t0 * xstep;
      // ---- (2) re-run the state recursion through the segment.  Fully unrolled (CK - 1 steps) so that the rotating buffer of
      // observation rows xr[row % 4] has static indices: row j + 3 is requested while step j runs (the L2 round trip is
      // longer than one of these short steps).  Leaves x_{t0 + nst - 1} in x[1] for the first step of the walk.
      float* sp = slot0;
      {
        f32x2 cP[NPA][R], xrP[4][NPA][D];
        float cS[R], xrS[4][D];
        CB::template load<false>(sp + lp, sp + ls, cP, cS);
        XB::template load<true>(xsp, xss, xrP[0], xrS[0]);
        if (nst > 1) XB::template load<true>(xsp + xstep, xss + xstep, xrP[1], xrS[1]);
        if (nst > 2) XB::template load<true>(xsp + 2 * xstep, xss + 2 * xstep, xrP[2], xrS[2]);
        static_for<0, CK - 1>([&](auto QC) {
          constexpr int q = decltype(QC)::value;
          if (q + 1 < nst) {
            if (q + 3 < nst) XB::template load<true>(xsp + (q + 3) * xstep, xss + (q + 3) * xstep, xrP[(q + 3) % 4], xrS[(q + 3) % 4]);
            const float* r = chunk + q * DM::REC;
            auto run = [&](const auto& rr) {
              LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2)
                Trial<DM>::template advance<f32x2>(rr, xrP[q % 4][p2], xrP[(q + 1) % 4][p2], cP[p2]);
              if constexpr (NS) Trial<DM>::template advance<float>(rr, xrS[q % 4], xrS[(q + 1) % 4], cS);
            };
            if constexpr (rec_in_regs<DM>() && LQGK_REV_REC_REGS) {
              RecRegs<DM> rr;
              rr.load(r);
              run(rr);
            } else {
              run(r);
            }
            sp = next_slot(sp);
            CB::store(sp + lp, sp + ls, cP, cS);
          }
        });
        static_for<0, CK>([&](auto JC) {             // x_{t0 + nst - 1}: static for full segments, selected for the ragged last one
          constexpr int j = decltype(JC)::value;
          if (nst - 1 == j) {
            LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) LQGK_UNROLL for (int m = 0; m < D; ++m) xP[1][p2][m] = xrP[j % 4][p2][m];
            LQGK_UNROLL for (int m = 0; m < D; ++m) xS[1][m] = xrS[j % 4][m];
          }
        });
      }
      // ---- (3) walk the segment backwards; sp = slot of its last step
      const float* xqp = xsp + (size_t)(nst - 1) * xstep;   // row of the step being processed; walks down one row per step
      const float* xqs = xss + (size_t)(nst - 1) * xstep;
      auto step = [&](auto PC, int q, bool top) {
        constexpr int P = decltype(PC)::value, Q = P ^ 1;
        const float* r = chunk + q * DM::REC;
        f32x2 cP[NPA][R];
        float cS[R];
        CB::template load<false>(sp + lp, sp + ls, cP, cS);
        f32x2 eP[NPA][D], vP[NPA][D], wvP[NPA][D], nebP[NPA][D];
        float eS[D], vS[D], wvS[D], nebS[D];
        auto run = [&](const auto& rr) {
          LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2)
            Trial<DM>::template rev<f32x2>(rr, xP[P][p2], xP[Q][p2], cP[p2], wP[p2], cbP[P][p2], eP[p2], vP[p2], wvP[p2], nebP[p2], cbP[Q][p2]);
          if constexpr (NS) Trial<DM>::template rev<float>(rr, xS[P], xS[Q], cS, wS, cbS[P], eS, vS, wvS, nebS, cbS[Q]);
        };
        if constexpr (rec_in_regs<DM>() && LQGK_REV_REC_REGS) {
          RecRegs<DM> rr;
          rr.load(r);
          run(rr);
        } else {
          run(r);
        }
        xqp -= xstep;
        xqs -= xstep;
        if (q > 0) {
          // x_{t-1} for the next step, requested only after this step's residuals exist (the empty asm makes the row pointer
          // depend on them): x_{t+1} in x[Q] is dead by then, so the loads land in its registers and no copy is needed
          if constexpr (NP > 0) asm volatile("" : "+l"(xqp) : "l"(Ops<f32x2>::u(eP[0][0])));
          else asm volatile("" : "+l"(xqs) : "f"(eS[0]));
          XB::template load<true>(xqp, xqs, xP[Q], xS[Q]);
        }
        if (top && k > ka) {
          // the slot of the segment's last step has been consumed (its values are operands of the arithmetic above):
          // the checkpoint of the next segment to process lands there while this one is walked
          hkp -= hstep;
          hks -= hstep;
          CB::copy_async(sp + lp, sp + ls, hkp, hks);
          slot0 = sp;
        }
        auto term = [&](auto IDXC) -> float {
          constexpr int IDX = decltype(IDXC)::value;
          float a = 0.f;
          if constexpr (NP > 0) {
            f32x2 acc = f32x2{0.f, 0.f};
            LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2)
              acc = Trial<DM>::template sum_acc<IDX, f32x2>(acc, cbP[P][p2], nebP[p2], xP[P][p2], cP[p2], eP[p2], vP[p2], wvP[p2]);
            a = acc.x + acc.y;
          }
          if constexpr (NS) a = Trial<DM>::template sum_acc<IDX, float>(a, cbS[P], nebS, xS[P], cS, eS, vS, wvS);
          return a;
        };
        static_for<0, NFULL>([&](auto G) {
          float val[32];
          static_for<0, 32>([&](auto J) {
            val[decltype(J)::value] = term(std::integral_constant<int, decltype(G)::value * 32 + decltype(J)::value>{});
          });
          float4* dst = reinterpret_cast<float4*>(red + lane * TRIAL_RED_STRIDE);
          LQGK_UNROLL for (int q4 = 0; q4 < 8; ++q4) dst[q4] = make_float4(val[4 * q4], val[4 * q4 + 1], val[4 * q4 + 2], val[4 * q4 + 3]);
          __syncwarp();
          float part[4] = {0.f, 0.f, 0.f, 0.f};
          LQGK_UNROLL for (int k2 = 0; k2 < 32; ++k2) part[k2 & 3] += red[k2 * TRIAL_RED_STRIDE + lane];
          const float tot = (part[0] + part[1]) + (part[2] + part[3]);
          __syncwarp();
          const int idx = decltype(G)::value * 32 + lane;
          if (blk == 0) out[idx] = tot;
          else out[idx] += tot;
        });
        if constexpr (REM > 0) {
          float val[VREM];
          static_for<0, VREM>([&](auto J) { val[decltype(J)::value] = term(std::integral_constant<int, NFULL * 32 + decltype(J)::value>{}); });
          float tot = warp_transpose_reduce<VREM>(val, lane);
          const int vi = lane / (32 / VREM);
          const int idx = NFULL * 32 + vi;
          if ((lane % (32 / VREM)) == 0 && idx < DM::SUMP) {
            if (blk == 0) out[idx] = tot;
            else out[idx] += tot;
          }
        }
        out -= DM::SUMP;
        sp = prev_slot(sp);
      };
      {
        int q = nst - 1;
        bool top = true;
#pragma unroll 1
        while (true) {
          step(std::integral_constant<int, 1>{}, q, top);
          top = false;
          if (--q < 0) {
            // odd number of steps (ragged last segment, odd CK): put the carried state back where a walk starts from
            LQGK_UNROLL for (int p2 = 0; p2 < NP; ++p2) {
              LQGK_UNROLL for (int m = 0; m < R; ++m) cbP[1][p2][m] = cbP[0][p2][m];
              LQGK_UNROLL for (int m = 0; m < D; ++m) xP[0][p2][m] = xP[1][p2][m];
            }
            if constexpr (NS) {
              LQGK_UNROLL for (int m = 0; m < R; ++m) cbS[1][m] = cbS[0][m];
              LQGK_UNROLL for (int m = 0; m < D; ++m) xS[0][m] = xS[1][m];
            }
            break;
          }
          step(std::integral_constant<int, 0>{}, q, false);
          if (--q < 0) break;
        }
      }
      __syncwarp();
      if (kk + 2 < nloc) ring.issue(kb - 1 - (kk + 2), st);
    }
    if (ka > 0) CB::store(carp, cars, cbP[1], cbS[1]);   // cotangent of c_{ka CK} for the launch that continues below
  }
}

}  // namespace lqgk
