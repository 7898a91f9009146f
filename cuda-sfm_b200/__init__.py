"""sfm-b200: B200-native RANSAC essential matrix -> pose -> triangulation.

The directory name carries a hyphen (it mirrors the reference's repo name), so
import it through ``__graft_entry__.load_package()`` or put the repo root on
sys.path and use ``importlib`` - it registers itself as ``cuda_sfm_b200``.

The product path is the C-ABI CUDA library ``libsfmb200.so`` (include/sfmb200.h).
There is no CPU fallback: loading fails loudly when the library is missing.
"""
from .binding import Lib, SfmError, load_library, lib_path  # noqa: F401
from .image_pair import ImagePair, BatchedPairs, check_offsets, pack_ragged, unpack_ragged  # noqa: F401
from . import sharding, synthetic  # noqa: F401

__all__ = ["Lib", "SfmError", "load_library", "lib_path", "ImagePair", "BatchedPairs", "check_offsets", "pack_ragged", "unpack_ragged"]
