"""rayhs_b200 — B200-native (sm_100a CUDA) ray-casting path of RayHs behind a C ABI.

See DESIGN.md.  The Python layer mirrors the reference's interface for this path
(`Rendering`, `rayTrace`, `distributedRayTrace`, `writePPM`); the kernels live in
csrc/kernels.cu and are reached through librayhs_b200.so (include/rayhs_b200.h).
"""
from .host import (HIT_DTYPE, Accumulator, AdaptiveAccumulator, Features, Hits, Image, LightGroups, PeerFrames, Radiance, Rendering, Scene, Views, assemble_bands, buildRendering, closestIntersection, distributedRayTrace, init, main,
                   adaptiveRayTrace, progressiveRayTrace, rayTrace, shadowIntersection, traceRay,
                   render, renderFeatures, renderLightGroups, renderViews, render_device, render_multi, multi_shutdown, renderingFromScene, sample_offsets, scene_setup_ms, shard_global_rows, shutdown, sphereLight, thinLens, writePPM)

__all__ = ["HIT_DTYPE", "Accumulator", "AdaptiveAccumulator", "Features", "Hits", "Image", "LightGroups", "PeerFrames", "Radiance", "Rendering", "Scene", "Views", "assemble_bands", "buildRendering", "closestIntersection",
           "adaptiveRayTrace", "distributedRayTrace", "init", "main", "progressiveRayTrace", "rayTrace", "shadowIntersection", "traceRay", "render", "renderFeatures", "renderLightGroups", "renderViews", "render_device", "render_multi", "multi_shutdown", "renderingFromScene", "sample_offsets", "scene_setup_ms", "shard_global_rows", "shutdown",
           "sphereLight", "thinLens", "writePPM"]
