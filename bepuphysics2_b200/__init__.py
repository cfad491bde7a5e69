"""bepuphysics2_b200 — B200-native constraint solver + integrator behind bepuphysics2's solver surface.

The product is `libbepucuda.so` (hand-written sm_100a CUDA kernels behind the C ABI in include/bepucuda.h). This package
only holds what the hot path needs: the native sources (csrc/), their in-tree build, a ctypes view of the C ABI, the
host-side mirror of the reference's Simulation/Solver/Timestepper slice, and seeded scene generators for the benchmark configs.

There is no CPU fallback: creating a `CudaTimestepper` without a usable CUDA device raises.
"""
from .native import (  # noqa: F401
    BepuCudaError,
    CudaTimestepper,
    IntegratorDesc,
    ShapeLibrary,
    Simulation,
    Timings,
    load_libraries,
    type_info,
)

__all__ = ["BepuCudaError", "CudaTimestepper", "IntegratorDesc", "ShapeLibrary", "Simulation", "Timings", "load_libraries", "type_info"]
