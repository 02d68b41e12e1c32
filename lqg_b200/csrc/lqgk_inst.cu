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
int Runner<DMI>::run_f32(const Call& c) { return run<DMI, float>(c); }
template <>
int Runner<DMI>::run_f64(const Call& c) { return run<DMI, double>(c); }
template <>
size_t Runner<DMI>::plan_bytes(const LqgkDims& d, int mode, int32_t max_chunk) {
  size_t Sc = choose_chunk<DMI>(d, mode, false, (size_t)-1, max_chunk);
  return make_plan<DMI>(d, mode, false, Sc).bytes;
}
#if !defined(LQGK_BIG)   // (the dimension dispatch hands the SDN paths small tuples only)
template <>
int Runner<DMI>::run_sdn(const SdnArgs& a, cudaStream_t st) {
  k_sdn_gains<DMI><<<(a.S + 31) / 32, 32, 0, st>>>(a);
  LQGK_LAUNCH_CHECK();
  return LQGK_OK;
}
template <>
int Runner<DMI>::run_sdn_loglik(const SdnLikArgs& a, bool f64, cudaStream_t st) { return launch_sdn_loglik<DMI>(a, f64, st); }
#endif
}  // namespace lqgk
