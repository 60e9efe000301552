"""slamrs_b200 -- B200-native grid particle-filter SLAM step behind slamrs' GridMapSlam API.

The compute path is libslamrs_gpu.so (hand-written sm_100a CUDA behind include/slamrs_gpu.h).
This package is the host-side mirror of the reference interface plus the synthetic-input
generator. Importing it never falls back to a CPU implementation.
"""
from .slam import (Clustering, GpuPlacement, GridData, GridMapLocalizer, GridMapSlam, GridMapSlamConfig, Kld, Measurement, Observation,
                   Odometry, Pose, Recovery, ScanMatcher, SensorModel, grid_cells, nccl_unique_id)

__all__ = ["Clustering", "GpuPlacement", "GridData", "GridMapLocalizer", "GridMapSlam", "GridMapSlamConfig", "Kld", "Measurement",
           "Observation", "Odometry", "Pose", "Recovery", "ScanMatcher", "SensorModel", "grid_cells", "nccl_unique_id"]
