"""pcreg_b200 -- B200-native (sm_100a) implementation of PCReg's alignment hot path.

Everything computes in libpcreg_b200.so (hand-written CUDA behind the C ABI of include/pcreg.h);
this package is only the host-side mirror of the reference's MATLAB interface.  No CPU fallback.
"""
from ._lib import PcregError, init, shutdown, load, LIB_PATH  # noqa: F401
from .api import (  # noqa: F401
    Model, cloud_normals, getLocalPoints, getLocalPoints_batch, getSpacialHistogramDescriptors, spatial_histogram_edges, AlignPoints, AlignPoints_KNN, AlignPoints_knn, AlignPoints_weighted, AlignPoints_c,
    AlignPoints_KNN_c, align_points_batch, estimateTransform, estimate_transform_batch, ransac, ransac_seeded, ransac_batch,
    getMatches, transfer_colors, quickTF, TF_FORWARD, TF_INVERT, TF_MRDIVIDE, icp_batch, icp_batch_windows, icp_covariance, icp_covariance_windows, icp_opts, icp_stop, icp_extrap, set_profiling, last_profile, launch_count,
    NN_BRUTE, NN_GRID, METRIC_SAD, METRIC_SSD, ICP_PLAIN, ICP_KNN, ICP_WEIGHTED, ICP_POINT_TO_POINT, ICP_POINT_TO_PLANE, ICP_PLANE_TO_PLANE,
    ALIGN_PLAIN, ALIGN_KNN_FRAC, ALIGN_KNN_ABS, ALIGN_WEIGHTED, ALIGN_C, ALIGN_KNN_C,
)


def device_count() -> int:
    """Devices selected by the last init() (pcreg_device_count)."""
    return int(load().pcreg_device_count())
