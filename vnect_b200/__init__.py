"""vnect_b200 -- B200-native (sm_100a) implementation of the VNect per-frame hot path.

Public surface: ``VNectEstimator`` (drop-in for the reference class, src/estimator.py:16-142) and ``VNectEngine`` (the
batched multi-stream form).  The compute lives in ``lib/libvnect_b200.so`` (hand-written CUDA: tcgen05/TMEM/TMA
implicit-GEMM convolutions, fused pre- and post-processing); this package only marshals pointers through ctypes.
"""
from .estimator import ORIENTATIONS, Joints2Angles, VNectEngine, VNectEstimator  # noqa: F401
from .hog_box import HOGBox  # noqa: F401

__all__ = ["VNectEstimator", "VNectEngine", "Joints2Angles", "HOGBox", "ORIENTATIONS"]
