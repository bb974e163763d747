"""ri_b200 — B200-native (sm_100a) front end of the rotation-invariant PVCNN feature extractor.

Importable as `ri_b200` (see /ri_b200.py at the repo root; the directory name carries the reference's full name).
Layout:
    csrc/           hand-written CUDA kernels + the C ABI of include/ri_b200.h  -> libri_b200.so
    _lib.py         ctypes binding (raises if the library is missing: there is no fallback path)
    ops.py          torch custom ops  torch.ops.ri.*
    backend.py      `_backend` with the reference pybind module's function names (drop-in boundary)
    functional/     the reference's PVCNN.modules.functional hot-path API
    modules/        the reference's PVCNN.modules hot-path classes (Voxelization, Spherical_Voxelization, knnModule, PVConv)
    frontend.py     the fused, graph-captured front-end engine (what bench.py measures)
    matcher.py      mutual-nearest-neighbour descriptor matching
    registration.py matches -> RANSAC / Kabsch pose -> RRE / RTE / RMSE meter (the reference's registration meter)
    subsampling.py  barycentre grid subsampling (the reference's utils/grid_subsampleing.py API) and the farthest-point
                    bridge from its variable-length output to a fixed-size batch
    shard.py        one-process-per-GPU sharding helpers
    synth.py        seeded synthetic inputs
"""
from . import _lib            # noqa: F401  raises ImportError when libri_b200.so has not been built
from . import ops             # noqa: F401  registers torch.ops.ri.*
from .backend import _backend  # noqa: F401
from . import functional, modules  # noqa: F401
from .frontend import FrontEnd, FrontEndLanes, FrontEndPipeline  # noqa: F401
from . import shard, synth, matcher, subsampling, registration  # noqa: F401
from .subsampling import grid_sub_sampling, grid_sub_sampling_many, farthest_point_batch  # noqa: F401

__version__ = '0.1.0'
