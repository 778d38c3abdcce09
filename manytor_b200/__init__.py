"""manytor_b200 -- B200-native batched implementation of ManyTor's step loop.

    import manytor_b200.manytor as tor      # drop-in for the reference's manytor.py
    from manytor_b200 import BatchedEnvs    # device-tensor API over the C ABI

The compute lives in manytor_b200/lib/libmanytor_b200.so (CUDA, sm_100a),
declared in include/manytor_b200.h.  There is no CPU fallback.
"""
from ._lib import MantorLibraryError, library_path, load as load_library  # noqa: F401
from .core import ArmSpec, BatchedEnvs, Branches, FinalInfo, REFERENCE_ARM, Trajectory, UR5_ARM  # noqa: F401
from . import distributed  # noqa: F401
from .vector_env import ManyTorVectorEnv  # noqa: F401

__all__ = ["ArmSpec", "BatchedEnvs", "Branches", "FinalInfo", "REFERENCE_ARM", "Trajectory", "UR5_ARM", "MantorLibraryError",
           "library_path", "load_library", "distributed", "ManyTorVectorEnv"]
