"""ekf-slam_b200 — B200-native batched 1-point-RANSAC EKF-SLAM filter step.

Public surface:
  * :class:`FilterBank` (bank.py)     — B filters resident on one GPU, stage-by-stage or fused step
  * api.py                            — the reference's function names on `filter` / `features_info`
  * synth.py                          — synthetic point-field sequences (workload generator)
  * sharding.py                       — one process per GPU, filters partitioned across ranks
The compute path is libekfslam.so (csrc/, C ABI in include/ekfslam.h); there is no CPU fallback.
"""
from ._lib import (EkfSlamError, FEAT_NONE, FEAT_INVERSEDEPTH, FEAT_CARTESIAN,  # noqa: F401
                   F_HAS_H, F_HAS_Z, F_IC, F_LI, F_HI, F_CAND, LIB_PATH,
                   EVAL_FIELDS, EVAL_CAM_NOT_SPD, EVAL_NO_TRUTH, EVAL_NOT_EVALUABLE)
from .bank import FilterBank  # noqa: F401

__version__ = "0.1.0"
