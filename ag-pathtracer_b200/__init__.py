"""ag-pathtracer_b200: B200-native (sm_100a) implementation of ag-pathtracer's per-pixel
path-tracing hot path.

Layout: ``csrc/`` CUDA kernels + C ABI (``libagpt.so``), ``host/`` C++ mirror of the reference's
scene API (``libagpt_host.so``), ``binding.py`` ctypes harness binding.  The directory name has
a hyphen, so tests and bench load this package through ``importlib`` under the module name
``agpt_b200`` (see ``tests/conftest.py`` / ``__graft_entry__.py``).
"""
from .binding import (AgptError, Context, Group, HostScene, HostTracer, Material, Stats, FLAG_COUNTERS, FLAG_TIMING,  # noqa: F401
                      FLAG_STRICT_BOXES, MAT_DISNEY, MAT_MIRROR, MAT_GLASS, LOBE_GLASS_REFLECT, LOBE_GLASS_TRANSMIT, HIT_DTYPE, config_defaults, core, device_count, host,
                      lib_paths, make_material, pinned_film, set_build_options, get_build_options, RawMesh, MeshDesc, FLAG_RAYS_FINAL, FLAG_RR_BY_BOUNCE,
                      PRIM_DTYPE, SPHERE_DTYPE, PLANE_DTYPE, LIGHT_DTYPE, NODE_DTYPE, PRIM_SPHERE, PRIM_PLANE, PRIM_BVH_MESH, PRIM_MESH, PRIM_INSTANCE,
                      LIGHT_AREA, LIGHT_UNIFORM_INFINITE, LIGHT_INFINITE_AREA, LIGHT_SAMPLE_SHAPE, Adaptive, adaptive, DenoiseParams,
                      denoise_params, ReprojectParams, reproject_params, MaterialTextures, material_textures,
                      AlphaMask, alpha_mask, Emission, emission)
from . import multigpu  # noqa: F401,E402
