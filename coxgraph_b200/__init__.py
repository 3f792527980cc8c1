"""coxgraph_b200 — B200-native TSDF fusion engine for coxgraph's hot path.

The product is the C-ABI shared library (include/coxgraph_b200.h, built from csrc/ into
lib/libcoxgraph_b200.so); `api` mirrors the reference-facing interface on top of it and `synth`
generates the synthetic depth streams of the benchmark.  Nothing here falls back to the CPU.
"""
from . import capi  # noqa: F401
from .api import (Context, Layer, depthCamera, esdfConfig, TsdfIntegrator, TsdfIntegratorConfig,  # noqa: F401
                  getProjectedMap, mergeLayerAintoLayerB, meshToFrames, recoverMesh,
                  reprojectSubmaps, VOXEL_DTYPE)
