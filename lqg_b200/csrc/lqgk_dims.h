// lqgk_dims.h -- the compiled (x, b, u, y, d) instantiations: dynamics state, belief state, control,
// observation, observed-by-experimenter dims.  One line per reference model family (lqg/tracking/*.py).
#pragma once
// clang-format off
#define LQGK_FOR_EACH_DIMS(M)                                                                       \
  M(2, 2, 1, 2, 2)   /* BoundedActor / OptimalActor dim=1 (basic.py:43-87)            [config c1] */ \
  M(2, 2, 1, 1, 2)   /* RelativeObservationBoundedActor dim=1 (basic.py:90-124)                   */ \
  M(2, 3, 1, 2, 2)   /* SubjectiveActor dim=1 (subjective.py:15-47)                               */ \
  M(4, 4, 2, 4, 4)   /* BoundedActor dim=2                                                        */ \
  M(4, 4, 2, 2, 4)   /* RelativeObservationBoundedActor dim=2                                     */ \
  M(4, 6, 2, 4, 4)   /* SubjectiveActor dim=2                               [configs c2, c3, c5] */ \
  M(4, 4, 1, 3, 2)   /* PointMassBoundedActor, observed target+cursor (point_mass.py, main.py:51) */ \
  M(5, 5, 1, 2, 2)   /* HandMotionModelTrackingTask (notebooks/HandModel.ipynb): target + pos/vel/force/act. */ \
  M(6, 6, 1, 2, 2)   /* TemporalDelayModel(BoundedActor dim=1, delay=2) (delay.py:9-41): motor-delay family */ \
  M(12, 12, 1, 3, 2) /* TemporalDelayModel(PointMassBoundedActor, delay=2): 12-dim state, joint dim 24 [config c4]; large-system kernels (lqgk_bigw.cuh) */
// Tuples compiled ONLY for the all-FP64 per-trial likelihood (k_sdn_loglik: lqgk_sdn_loglik_*, System.log_likelihood_fp64): models
// whose innovation covariance is too ill-conditioned for the FP32 per-trial arithmetic of the main path (DESIGN.md section 7).
#define LQGK_FOR_EACH_FP64_ONLY_DIMS(M)                                                                      \
  M(4, 4, 1, 3, 4)   /* PointMassBoundedActor with all four states observed (point_mass.py:7-47; condition number ~1e9) */
// clang-format on
