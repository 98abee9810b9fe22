"""nav-slam_b200 -- B200-native (sm_100a CUDA) implementation of NAV-SLAM's data-parallel front end.

Layout:
  csrc/    CUDA kernels + the C ABI (include/navslam_b200.h) -> _build/libnavslam_b200.so
  shim/    per-shape shim exporting the reference's own symbols (include/navslam_ref_abi.h)
  build.py nvcc / gcc build recipe (in-tree, sm_100a only)
  binding.py  ctypes caller used by tests, bench.py and smoke()
  synth.py    seeded synthetic inputs of the five BASELINE.json configs
  sharding.py multi-GPU partitioning (independent sequences, query sharding)

The directory name has a hyphen, so import it with importlib.import_module("nav-slam_b200").
"""
from . import build, synth  # noqa: F401
from .binding import (Context, KdTree, NavError, bruteforce_nn_dev, csv_format_frame,  # noqa: F401
                      device_count, fit_from_stats, imu_json_read, l5_json_read, l9_csv_read, l9_csv_read_mm,
                      load_library, to_mm)
