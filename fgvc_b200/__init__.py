"""fgvc_b200 -- B200-native label propagation for FGVC (mmpt): hand-written sm_100a
kernels behind a C ABI, host side mirroring the reference's operator / tracker / test API.
"""
from ._lib import ENGINE_AUTO, ENGINE_SIMT, ENGINE_TCGEN05, FgvcError  # noqa: F401
from .ops import (compute_affinity, masked_attention_efficient, masked_attention_efficient_c2f,  # noqa: F401
                  masked_attention_efficient_v2, propagate, propagate_temporal, spatial_neighbor)
from .tracker import B200HRVanillaTracker, B200VanillaTracker, HRVanillaTracker, VanillaTracker  # noqa: F401
from .c2f_tracker import B200C2FTracker, C2FPointTracker, C2FTracker  # noqa: F401
from .apis import (DistributedSampler, collect_results_cpu, collect_results_gpu,  # noqa: F401
                   multi_gpu_test, sharded_forward_test, single_gpu_test)

__version__ = "0.1.0"
