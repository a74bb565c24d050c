"""tft_vs_fund_b200 -- B200-native batched linear three-view pose estimation.

Drop-in for the linear hot path of LauraFJulia/TFT_vs_Fund: the functions below
carry the reference's names and signatures and run entirely in hand-written
CUDA (sm_100a) behind the C ABI of ``include/tvf.h`` (``libtvf.so``).  There is
no CPU fallback; importing is cheap, the library is loaded on first use.
"""
from .api import (  # noqa: F401
    LinearTFTPoseEstimation, LinearFPoseEstimation, OptimFPoseEstimation, linearTFT, linearF, optimF,
    Normalize2Ddata, transform_TFT, R_t_from_TFT, TFT_from_P, triangulation3D,
    ReprError, AngError, crossM, project3Dpoints, PoseResult, bundle_adjust, BundleAdjustResult,
    ba_covariance, CovarianceResult, pose_rms_errors, consensus, ransac_pose, RansacResult,
)
from ._lib import TvfError, Handle, handle, load, LIB_PATH  # noqa: F401
from .scene import generateSyntheticScene, sweep_batch, SceneRNG  # noqa: F401
from . import experiments, sharding, epfl  # noqa: F401

__all__ = [
    "LinearTFTPoseEstimation", "LinearFPoseEstimation", "OptimFPoseEstimation", "linearTFT", "linearF", "optimF",
    "Normalize2Ddata", "transform_TFT", "R_t_from_TFT", "TFT_from_P",
    "triangulation3D", "ReprError", "AngError", "crossM", "project3Dpoints", "bundle_adjust",
    "ba_covariance", "pose_rms_errors", "consensus", "ransac_pose",
    "generateSyntheticScene", "sweep_batch", "Handle", "handle", "TvfError",
]
