// lqgk_inst.cu -- instantiates every kernel and the launch sequence for ONE dimension tuple, selected with
// -DLQGK_INST_X/B/U/Y/D (one object file per line of lqgk_dims.h; __graft_entry__.build() compiles them in parallel).
#include "lqgk_run.cuh"

#if !defined(LQGK_INST_X)
#error "compile with -DLQGK_INST_X=.. -DLQGK_INST_B=.. -DLQGK_INST_U=.. -DLQGK_INST_Y=.. -DLQGK_INST_D=.."
#endif

namespace lqgk {
using DMI = Dims<LQGK_INST_X, LQGK_INST_B, LQGK_INST_U, LQGK_INST_Y, LQGK_INST_D>;
#if defined(LQGK_BIG)
static_assert(is_big<DMI>(), "-DLQGK_BIG is for joint dims > 12 only");
#else
static_assert(!is_big<DMI>(), "joint dims > 12 must be compiled with -DLQGK_BIG");
#endif
template <>
int Runner<LQGK_INST_X, LQGK_INST_B, LQGK_INST_U, LQGK_INST_Y, LQGK_INST_D>::run_f32(const Call& c) { return run<DMI, float>(c); }
template <>
int Runner<LQGK_INST_X, LQGK_INST_B, LQGK_INST_U, LQGK_INST_Y, LQGK_INST_D>::run_f64(const Call& c) { return run<DMI, double>(c); }
template <>
size_t Runner<LQGK_INST_X, LQGK_INST_B, LQGK_INST_U, LQGK_INST_Y, LQGK_INST_D>::plan_bytes(const LqgkDims& d, int mode, int32_t max_chunk) {
  size_t Sc = choose_chunk<DMI>(d, mode, false, (size_t)-1, max_chunk);
  return make_plan<DMI>(d, mode, false, Sc).bytes;
}
template <>
int Runner<LQGK_INST_X, LQGK_INST_B, LQGK_INST_U, LQGK_INST_Y, LQGK_INST_D>::run_sdn(const SdnArgs& a, cudaStream_t st) {
#if defined(LQGK_BIG)
  (void)a; (void)st;
  return LQGK_E_UNSUPPORTED;
#else
  k_sdn_gains<DMI><<<(a.S + 31) / 32, 32, 0, st>>>(a);
  LQGK_LAUNCH_CHECK();
  return LQGK_OK;
#endif
}
template <>
int Runner<LQGK_INST_X, LQGK_INST_B, LQGK_INST_U, LQGK_INST_Y, LQGK_INST_D>::run_sdn_loglik(const SdnLikArgs& a, bool f64, cudaStream_t st) {
#if defined(LQGK_BIG)
  (void)a; (void)f64; (void)st;
  return LQGK_E_UNSUPPORTED;
#else
  const size_t total = (size_t)a.S * a.N;
  const unsigned blocks = (unsigned)((total + 63) / 64);
  if (f64) k_sdn_loglik<DMI, double><<<blocks, 64, 0, st>>>(a);
  else k_sdn_loglik<DMI, float><<<blocks, 64, 0, st>>>(a);
  LQGK_LAUNCH_CHECK();
  return LQGK_OK;
#endif
}
}  // namespace lqgk
