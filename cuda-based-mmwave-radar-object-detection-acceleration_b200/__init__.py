"""B200-native mmWave radar processing chain (int16 ADC cube -> detections).

The product is libmmw_radar_b200.so (hand-written sm_100a CUDA behind the C ABI of
include/mmw_radar.h and the reference's own cudaProcessing() entry point, include/mmw_legacy.h).
This package holds its sources (csrc/), the in-tree build recipe, the ctypes binding that mirrors
the C ABI one to one, the frame-sharding / gather plumbing and the synthetic capture generator.

The directory name contains hyphens (it mirrors the reference repository's name), so import it
through `__graft_entry__.load_package()` or importlib, not with an `import` statement.
"""
from . import api, build, sharding, synth  # noqa: F401
from .api import DET_DTYPE, OBJ_DTYPE, TARGET_DTYPE, PeerExchange, RadarContext, RadarError, RadarGroup, RadarParams, cudaProcessing  # noqa: F401
