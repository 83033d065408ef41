"""B200-native path-tracing hot path of mu-lambda/mu-lambda-raytracer.

The product is `librt_b200.so` (hand-written CUDA for sm_100a behind the C ABI of include/rt_b200.h).  This
package is the thin Python host layer over that ABI, mirroring the reference's own interface for the path
(`worlds()`, `Camera`, `RenderingParams`, `RecursiveRayTracer`, `SeedableRngator`, `Renderer.new_with_rng(...)
.render(logger)`; src/raytrace.rs:137-198, src/worlds.rs:14-19, src/camera.rs:15-38).
"""
from . import abi  # noqa: F401
from .renderer import (BlackBackground, Camera, GradientBackground, RecursiveRayTracer, Renderer,  # noqa: F401
                       RenderingParams, Scene, SceneDescription, SeedableRngator, World, denoise, denoise_cross,
                       denoise_guided, denoise_sure, load_earthmap, to_ppm, worlds)
