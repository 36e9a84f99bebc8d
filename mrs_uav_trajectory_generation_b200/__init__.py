"""mrs_uav_trajectory_generation_b200 -- B200-native (sm_100a) batched polynomial trajectory optimiser.

Drop-in for the hot path of ctu-mrs/mrs_uav_trajectory_generation (the vendored eth_trajectory_generation QP, NLopt-style
segment-time allocation, analytic + sampled feasibility, dt-sampling) behind the C ABI of include/tg_b200.h.
The package holds only what that path needs: csrc/ (CUDA kernels + C ABI), the ctypes binding (_capi.py), the
reference-shaped host API (api.py), problem-index sharding for one process per GPU (sharding.py) and the synthetic
workloads of BASELINE.json (workloads.py).

There is no CPU implementation in this package: without libtg_b200.so and a CUDA device every entry point raises.
"""
from ._capi import Context, Library, Params, Result, RESULT_DTYPE, TgError, DEFAULT_LIB  # noqa: F401
from . import workloads  # noqa: F401
from . import sharding  # noqa: F401
from .api import (  # noqa: F401
    Vertex,
    PolynomialOptimization,
    PolynomialOptimizationNonLinear,
    NonlinearOptimizationParameters,
    Trajectory,
    sample_whole_trajectory,
    sample_trajectory_in_range,
    sample_trajectory_start_duration,
    sample_trajectories_in_range,
    estimate_segment_times,
    estimate_segment_times_euclidean,
    estimate_segment_times_baca,
    estimate_segment_times_batch,
    TrajectoryGenerator,
    derivative_order,
)

__version__ = "0.1.0"
