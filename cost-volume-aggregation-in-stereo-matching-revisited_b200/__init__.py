"""B200-native DCANet cost-volume hot path (feature maps -> disparity) behind the reference's module API."""
from . import (_lib, engine, evaluation, frontend, fusion, geometry, guide, gwcnet, hshard, kitti_io, occupancy,
               pipeline, stixel, tracking, wls)
from . import gwcnet_dca0_g, gwcnet_dca1_g, gwcnet_dca2_g, gwcnet_dca4_g
from .cva import Multi_Aggregation, cva
from .engine import LR_CONSISTENT, LR_MISMATCH, LR_OCCLUDED, LR_OUT_OF_VIEW, Confidence, LRCheck
from .evaluation import DisparityMeter, evaluate_files, read_kitti_disparity, read_pfm
from .fusion import Rendered, SurfacePoints, TSDFVolume, fuse_files, read_kitti_poses, save_kitti_poses
from .geometry import (PointCloud, StereoCalib, read_kitti_calib, read_middlebury_calib, reproject,
                       reproject_files, save_depth_png, save_ply)
from .guide import lidar_hints, read_velodyne
from .motion import Motion, MovingObjects, motion           # the function: the module is <package>.motion in sys.modules
from .occupancy import FREE, OCCUPIED, UNKNOWN, Agreement, OccupancyGrid
from .gwcnet_dca_g import GwcNet, feature_extraction, hourglass
from .pipeline import HotPathPipeline
from .rectify import (RectifyPipeline, Rectified, StereoRectifier, read_kitti_raw_rectifier, rectify,
                      rectify_files)
from .self_attention import SelfAttentionBlock
from .stixel import GroundProfile, StixelMetric, Stixels, ground_profile, stixels
from .semantic_level import SemanticLevelContext
from .tracking import TrackResult, Tracker, Trajectory, track_files
from .wls import Refined, wls_filter
from .submodule import (PropgationNet_4x, build_concat_volume, build_cost_planes, build_gwc_volume, convbn,
                        convbn_3d, disparity_regression, softmax_disparity_regression)


def lr_consistency(disp_left, disp_right, tau=1.0):
    """Left-right consistency check of two disparities obtained elsewhere, fp32 CUDA [B,H,W] or [B,1,H,W] in their own
    views -> LRCheck(disp_right, label, filled) shaped like disp_left (include/dca_b200.h section 8)."""
    label, filled, _ = engine.lr_consistency(disp_left, disp_right, tau)
    return LRCheck(disp_right, label, filled)


__all__ = ["GwcNet", "feature_extraction", "hourglass", "cva", "Multi_Aggregation", "SemanticLevelContext",
           "SelfAttentionBlock", "PropgationNet_4x", "build_gwc_volume", "build_concat_volume", "build_cost_planes",
           "disparity_regression", "softmax_disparity_regression", "convbn", "convbn_3d", "engine", "hshard", "kitti_io", "HotPathPipeline",
           "evaluation", "DisparityMeter", "evaluate_files", "read_pfm", "read_kitti_disparity", "Confidence",
           "LRCheck", "lr_consistency", "LR_CONSISTENT", "LR_OCCLUDED", "LR_MISMATCH", "LR_OUT_OF_VIEW", "geometry",
           "StereoCalib", "PointCloud", "read_kitti_calib", "read_middlebury_calib", "reproject", "reproject_files",
           "save_ply", "save_depth_png", "StereoRectifier", "read_kitti_raw_rectifier", "rectify", "Rectified",
           "RectifyPipeline", "rectify_files", "wls", "wls_filter", "Refined", "fusion", "TSDFVolume", "SurfacePoints",
           "fuse_files", "read_kitti_poses", "Rendered", "save_kitti_poses", "tracking", "Tracker", "TrackResult",
           "Trajectory", "track_files", "guide", "lidar_hints", "read_velodyne", "stixel", "ground_profile", "stixels",
           "GroundProfile", "Stixels", "StixelMetric", "motion", "Motion", "MovingObjects", "occupancy",
           "OccupancyGrid", "Agreement", "FREE", "OCCUPIED", "UNKNOWN"]
