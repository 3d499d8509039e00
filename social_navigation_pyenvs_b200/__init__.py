"""B200-native batched crowd-stepping engine: drop-in for the per-step human motion update of Social-Navigation-PyEnvs.

Python here is host glue only; every number is produced by the hand-written sm_100a kernels in csrc/ behind the C ABI of
include/snp_b200.h.  Importing the package does not need a GPU; calling into it does, and there is no CPU fallback.
"""
from .engine import CrowdEngine, SFMS, model_parameters  # noqa: F401
from .forces_parallel import update_humans_parallel  # noqa: F401
from .large import TiledCrowdEngine  # noqa: F401
