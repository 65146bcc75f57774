"""vo_b200 — B200-native (sm_100a) hot path of the RGB-D visual-odometry pipeline.

descriptor matching -> keypoint gather / depth back-projection -> PnP-RANSAC -> relative pose, as
hand-written CUDA behind a C ABI (include/vo_b200.h, libvo_b200.so), with the reference's own Python
interface on top (feature_extractors/*.get_matches, VisualOdometry.process_frame / computepose_3D_2D,
vo_runner.py + config/vo_params.yaml).  Import this package as `vo_b200` (see ../vo_b200.py).
"""
from . import _lib  # noqa: F401
from ._lib import (VO_METRIC_COSINE, VO_METRIC_L2, VO_MODE_MUTUAL, VO_MODE_NN, VO_MODE_RATIO, VO_MODE_RATIO_MUTUAL,  # noqa: F401
                   VO_MODE_THRESH, VO_MODE_THRESH_MUTUAL, VO_NORM_HAMMING, VO_NORM_L2_U8, VO_PREC_F16X1, VO_PREC_F16X3, VO_PREC_FP32_SIMT,
                   VO_PREC_TF32X1, VO_PREC_TF32X3, VO_ST_KP_OUT_OF_IMAGE, VO_ST_NO_MODEL, VO_ST_OK,
                   VO_ST_TOO_FEW_POINTS, VO_ST_BAD_INPUT, VO_PNP_THROUGHPUT, VO_PNP_REFERENCE, VoError)

__all__ = ["_lib", "ops", "synthetic", "sequence"]
