"""ctypes binding over the two in-tree shared libraries.

* ``libagpt.so``      -- CUDA kernels behind the C ABI of ``include/agpt.h`` (the product).
* ``libagpt_host.so`` -- host mirror of the reference's C++ scene API behind ``include/agpt_host.h``.

Python is only the test / benchmark harness language here: the reference is C++, and so is the
host side of the drop-in.  Nothing in this module computes on the CPU; every ``Context`` method
is one C-ABI call.  If ``libagpt.so`` is missing or no CUDA device can be opened the calls raise
``AgptError`` -- there is deliberately no fallback.
"""
import ctypes
import os
from ctypes import POINTER, byref, c_char_p, c_float, c_int, c_int32, c_int64, c_uint32, c_uint64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

FLAG_COUNTERS = 1
FLAG_TIMING = 2
FLAG_STRICT_BOXES = 4
FLAG_RAYS_FINAL = 8
FLAG_RR_BY_BOUNCE = 16

MAT_DISNEY = 1
MAT_MIRROR = 2
MAT_GLASS = 3          # extension: rough dielectric (make_material: color = Kr = Kt, `metallic` slot = eta)
LOBE_GLASS_REFLECT, LOBE_GLASS_TRANSMIT = 16, 32


class AgptError(RuntimeError):
    pass


class Material(ctypes.Structure):  # agpt_material
    _fields_ = [("type", c_int32), ("lobes", c_uint32), ("roughness", c_float), ("metallic", c_float),
                ("diffuse_r", c_float * 3), ("eta", c_float), ("spec_r0", c_float * 3), ("alpha_x", c_float),
                ("mirror_r", c_float * 3), ("alpha_y", c_float)]


class BvhNode(ctypes.Structure):  # agpt_bvh_node
    _fields_ = [("bmin", c_float * 3), ("bmax", c_float * 3), ("first", c_int32), ("count", c_int32)]


class MeshDesc(ctypes.Structure):  # agpt_mesh_desc
    _fields_ = [("nodes", c_void_p), ("n_nodes", c_int32), ("n_tris", c_int32), ("tri_verts", c_void_p), ("tri_ids", c_void_p),
                ("tri_normals", c_void_p), ("tri_uvs", c_void_p)]


PRIM_DTYPE = np.dtype([("type", np.int32), ("payload", np.int32), ("material", np.int32), ("area_light", np.int32)])        # agpt_prim
SPHERE_DTYPE = np.dtype([("center", np.float32, 3), ("r", np.float32), ("r2", np.float32), ("pad", np.float32, 3)])        # agpt_sphere
PLANE_DTYPE = np.dtype([("o", np.float32, 3), ("half_x", np.float32), ("half_z", np.float32), ("pad", np.float32, 3)])     # agpt_plane
# agpt_light; flags and pad share one sub-record so that rows written as (type, prim, (0, 0), lemit, 0) keep working
LIGHT_DTYPE = np.dtype([("type", np.int32), ("prim", np.int32), ("ext", [("flags", np.uint32), ("pad", np.float32)]), ("lemit", np.float32, 3),
                        ("pad2", np.float32)])
NODE_DTYPE = np.dtype([("bmin", np.float32, 3), ("bmax", np.float32, 3), ("first", np.int32), ("count", np.int32)])        # agpt_bvh_node
PRIM_SPHERE, PRIM_PLANE, PRIM_BVH_MESH, PRIM_MESH, PRIM_INSTANCE = 0, 1, 2, 3, 4
LIGHT_AREA, LIGHT_UNIFORM_INFINITE, LIGHT_INFINITE_AREA = 0, 1, 2
LIGHT_SAMPLE_SHAPE = 1     # agpt_light.flags (extension): next-event estimation samples the area light's plane or mesh


class RawMesh:
    """One agpt_mesh_desc built from numpy arrays (kept alive here): nodes = NODE_DTYPE array or None,
    tri_verts = [n, 3, 4] float32 (leaf order), tri_ids = [n] int32, optional normals [n, 3, 4] / uvs [n, 3, 2]."""

    def __init__(self, tri_verts, tri_ids=None, nodes=None, normals=None, uvs=None):
        self.verts = np.ascontiguousarray(tri_verts, np.float32).reshape(-1, 3, 4)
        n = len(self.verts)
        self.ids = np.ascontiguousarray(np.arange(n) if tri_ids is None else tri_ids, np.int32)
        self.nodes = None if nodes is None else np.ascontiguousarray(nodes, NODE_DTYPE)
        self.normals = None if normals is None else np.ascontiguousarray(normals, np.float32).reshape(n, 3, 4)
        self.uvs = None if uvs is None else np.ascontiguousarray(uvs, np.float32).reshape(n, 3, 2)

    def desc(self):
        ptr = lambda a: None if a is None else a.ctypes.data
        return MeshDesc(ptr(self.nodes), 0 if self.nodes is None else len(self.nodes), len(self.verts), ptr(self.verts), ptr(self.ids),
                        ptr(self.normals), ptr(self.uvs))


class Adaptive(ctypes.Structure):  # agpt_adaptive (extension: adaptive sampling)
    _fields_ = [("min_samples", c_int32), ("max_samples", c_int32), ("step", c_int32), ("tolerance", c_float), ("floor", c_float)]


def adaptive(min_samples, max_samples, step, tolerance, floor=0.0):
    """agpt_adaptive record; the convergence test it parameterises is stated in include/agpt.h and oracle/adaptive.py."""
    return Adaptive(int(min_samples), int(max_samples), int(step), float(tolerance), float(floor))


class DenoiseParams(ctypes.Structure):  # struct agpt_denoise (extension: the a-trous denoiser)
    _fields_ = [("iterations", c_int32), ("sigma_luminance", c_float), ("sigma_depth", c_float), ("normal_power_log2", c_int32)]


def denoise_params(iterations=5, sigma_luminance=8.0, sigma_depth=0.1, normal_power_log2=7):
    """struct agpt_denoise record; the filter it parameterises is stated in include/agpt.h and oracle/denoise.py.  The defaults
    are the best of tests/perf_denoise.py's sweep on cfg 3 at 16 spp and within 3 % of the best on cfg 5 (DESIGN.md section 10
    has the measurements)."""
    return DenoiseParams(int(iterations), float(sigma_luminance), float(sigma_depth), int(normal_power_log2))


class ReprojectParams(ctypes.Structure):  # agpt_reproject (extension: reprojection across camera moves)
    _fields_ = [("max_history", c_float), ("sigma_depth", c_float), ("min_normal_dot", c_float)]


def reproject_params(max_history=8.0, sigma_depth=0.05, min_normal_dot=0.5):
    """agpt_reproject record; the reprojection it parameterises is stated in include/agpt.h and oracle/reproject.py.  The defaults
    are the best of tests/perf_temporal.py's sweep on cfg 3 along a 16-frame orbit at 4 spp per frame and within 3 % of the best on
    cfg 5 (DESIGN.md section 10 has the measurements)."""
    return ReprojectParams(float(max_history), float(sigma_depth), float(min_normal_dot))


class Stats(ctypes.Structure):  # agpt_stats
    _fields_ = [(n, c_uint64) for n in ("paths", "rays_closest", "rays_shadow", "rays_mis", "rays_skip", "rays_mis_culled", "rays_tail_culled")] + \
               [(n, c_uint64 * 2) for n in ("node_visits", "box_tests", "tri_tests", "analytic_tests", "warp_steps", "lane_steps")] + \
               [(n, c_uint64) for n in ("kernel_launches", "launches_closest", "launches_any", "launches_shade", "waves")] + \
               [(n, c_float) for n in ("ms_render", "ms_trace_closest", "ms_trace_any", "ms_shade", "ms_other", "ms_reduce")] + \
               [("reduce_path", c_uint32)]

    def as_dict(self):
        d = {}
        for n, t in self._fields_:
            v = getattr(self, n)
            d[n] = list(v) if hasattr(v, "__len__") else v
        return d

    @property
    def rays(self):
        """Rays actually traced through the scene."""
        return self.rays_closest + self.rays_shadow + self.rays_mis

    @property
    def rays_reference_equivalent(self):
        """Rays the reference's PathTracer::Li issues for the same paths (traced + provably useless ones not traced)."""
        return self.rays + self.rays_mis_culled + self.rays_tail_culled

    def algorithmic_bytes(self, k):
        """SURVEY 8d: 64 B per interior visit + 48 B per triangle test + 32 B per analytic record
        + 64 B per ray (ray in, hit out, queue traffic).  k = 0 closest-hit kernel, 1 any-hit kernel."""
        rays = (self.rays_closest + self.rays_mis) if k == 0 else self.rays_shadow
        return 64 * self.node_visits[k] + 48 * self.tri_tests[k] + 32 * self.analytic_tests[k] + 64 * rays


class Texture(ctypes.Structure):      # agpt_texture
    _fields_ = [("width", c_int), ("height", c_int), ("rgb", POINTER(c_float))]


class MaterialTextures(ctypes.Structure):      # agpt_material_textures
    _fields_ = [("base", c_int32), ("roughness_metallic", c_int32), ("normal", c_int32), ("normal_scale", c_float), ("color", c_float * 3)]


def material_textures(base=-1, roughness_metallic=-1, normal=-1, normal_scale=1.0, color=(0.0, 0.0, 0.0)):
    """EXTENSION (agpt.h agpt_material_textures): one material's image bindings, indices into the images of
    Context.upload_material_textures or -1.  `color` is the base colour used where base is -1 and roughness_metallic is not."""
    return MaterialTextures(base, roughness_metallic, normal, normal_scale, (c_float * 3)(*color))


class AlphaMask(ctypes.Structure):      # agpt_alpha_mask
    _fields_ = [("texture", c_int32), ("channel", c_int32), ("cutoff", c_float), ("pad", c_int32)]


def alpha_mask(texture=-1, channel=0, cutoff=0.5):
    """EXTENSION (agpt.h agpt_alpha_mask): one material's cutout mask, channel `channel` (0, 1, 2) of resident texture `texture`
    (-1: no mask); the surface is there where that channel >= cutoff."""
    return AlphaMask(texture, channel, cutoff, 0)


class Emission(ctypes.Structure):       # agpt_emission
    _fields_ = [("texture", c_int32), ("factor", c_float * 3)]


def emission(texture=-1, factor=(0.0, 0.0, 0.0)):
    """EXTENSION (agpt.h agpt_emission): one material's emission, `factor` (linear RGB, finite, >= 0) times resident texture
    `texture` at the hit's uv, or `factor` alone for texture -1.  The material emits iff some factor component is > 0."""
    return Emission(texture, (c_float * 3)(*factor))


def _image_rows(images, who):
    imgs = [np.ascontiguousarray(a, np.float32) for a in images]
    for a in imgs:
        if a.ndim != 3 or a.shape[2] != 3:
            raise AgptError(f"{who}: every image must be an (H, W, 3) array")
    return imgs, (Texture * max(len(imgs), 1))(*[Texture(a.shape[1], a.shape[0], _fptr(a)) for a in imgs])


HIT_DTYPE = np.dtype([("found", np.uint32), ("prim", np.int32), ("tri", np.int32), ("t", np.float32)])

_core = None
_host = None


def lib_paths():
    # AGPT_LIB: experiment hook -- load an alternative build of the core library
    return os.environ.get("AGPT_LIB") or os.path.join(_HERE, "libagpt.so"), os.path.join(_HERE, "libagpt_host.so")


def core():
    """libagpt.so (loads without a GPU; every compute entry point then fails loudly)."""
    global _core
    if _core is None:
        path = lib_paths()[0]
        if not os.path.exists(path):
            raise AgptError(f"{path} is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU fallback)")
        lib = ctypes.CDLL(path, mode=ctypes.RTLD_GLOBAL)
        lib.agpt_last_error.restype = c_char_p
        _core = lib
    return _core


def host():
    global _host
    if _host is None:
        core()
        path = lib_paths()[1]
        if not os.path.exists(path):
            raise AgptError(f"{path} is not built")
        lib = ctypes.CDLL(path)
        lib.agpt_host_last_error.restype = c_char_p
        _host = lib
    return _host


def _check(rc, lib=None, host_side=False):
    if rc < 0:
        msg = (host().agpt_host_last_error() if host_side else core().agpt_last_error()) or b""
        raise AgptError(f"agpt error {rc}: {msg.decode(errors='replace')}")
    return rc


def _fptr(a):
    return a.ctypes.data_as(POINTER(c_float))


def device_count():
    n = c_int(0)
    rc = core().agpt_device_count(byref(n))
    return n.value if rc == 0 else 0


class Context:
    """agpt_ctx: one per GPU."""

    def __init__(self, device=0):
        self._h = c_void_p()
        _check(core().agpt_create(c_int(device), byref(self._h)))
        self.device = device
        self.width = self.height = 0

    def close(self):
        if self._h:
            core().agpt_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def set_stream(self, cuda_stream_ptr):
        _check(core().agpt_set_stream(self._h, c_void_p(cuda_stream_ptr)))

    # ---- raw table upload (what Scene::Flatten feeds the C ABI; tests build tables by hand) ----------
    def upload_meshes(self, meshes):
        descs = (MeshDesc * max(len(meshes), 1))(*[m.desc() for m in meshes])
        _check(core().agpt_upload_meshes(self._h, descs, c_int(len(meshes))))

    def upload_table(self, kind, rows):
        """kind in spheres / planes / primitives / materials / lights; rows = structured numpy array (or Material list)."""
        fn = getattr(core(), "agpt_upload_" + kind)
        if kind == "materials":
            arr = (Material * max(len(rows), 1))(*rows)
            _check(fn(self._h, arr, c_int(len(rows))))
            return
        dt = {"spheres": SPHERE_DTYPE, "planes": PLANE_DTYPE, "primitives": PRIM_DTYPE, "lights": LIGHT_DTYPE}[kind]
        rows = np.ascontiguousarray(rows, dt)
        _check(fn(self._h, rows.ctypes.data_as(c_void_p), c_int(len(rows))))

    def upload_instances(self, rows):
        """rows: structured array of agpt_instance records (mesh, pad[3], object_to_world[12], world_to_object[12])."""
        rows = np.ascontiguousarray(rows)
        assert rows.dtype.itemsize == 112
        _check(core().agpt_upload_instances(self._h, rows.ctypes.data_as(c_void_p), c_int(len(rows))))

    def upload_textures(self, images, material_texture):
        """EXTENSION (agpt.h agpt_upload_textures): images = base-colour textures, each a numpy (H, W, 3) float32 array of linear
        RGB, row 0 at v in [0, 1/H); material_texture[i] = index into images of material i's texture, or -1.  ([], []) clears."""
        imgs, rows = _image_rows(images, "upload_textures")
        mt = np.ascontiguousarray(material_texture, np.int32)
        _check(core().agpt_upload_textures(self._h, rows if imgs else None, c_int(len(imgs)),
                                           mt.ctypes.data_as(POINTER(c_int)) if mt.size else None, c_int(mt.size)))

    def upload_material_textures(self, images, bindings):
        """EXTENSION (agpt.h agpt_upload_material_textures): images as for upload_textures (normal maps and roughness-metallic maps
        are linear too); bindings[i] = material i's agpt.material_textures(...), a MaterialTextures row.  ([], []) clears."""
        imgs, rows = _image_rows(images, "upload_material_textures")
        bindings = list(bindings)
        for b in bindings:
            if not isinstance(b, MaterialTextures):
                raise AgptError("upload_material_textures: every binding must be a material_textures(...) row")
            if any(not -1 <= i < len(imgs) for i in (b.base, b.roughness_metallic, b.normal)):
                raise AgptError("upload_material_textures: a binding points outside the images")
            if not np.all(np.isfinite([b.normal_scale, *b.color])):
                raise AgptError("upload_material_textures: normal_scale and color must be finite")
        table = (MaterialTextures * max(len(bindings), 1))(*bindings)
        _check(core().agpt_upload_material_textures(self._h, rows if imgs else None, c_int(len(imgs)), table if bindings else None, c_int(len(bindings))))

    def upload_alpha_masks(self, bindings):
        """EXTENSION (agpt.h agpt_upload_alpha_masks): bindings[i] = material i's agpt.alpha_mask(...), naming a texture of the last
        texture upload.  [] clears.  A texture upload clears the masks."""
        bindings = list(bindings)
        for b in bindings:
            if not isinstance(b, AlphaMask):
                raise AgptError("upload_alpha_masks: every binding must be an alpha_mask(...) row")
            if b.texture < -1 or not 0 <= b.channel <= 2 or not np.isfinite(b.cutoff):
                raise AgptError("upload_alpha_masks: need texture >= -1, channel in [0, 2] and a finite cutoff")
        table = (AlphaMask * max(len(bindings), 1))(*bindings)
        _check(core().agpt_upload_alpha_masks(self._h, table if bindings else None, c_int(len(bindings))))

    def upload_emission(self, rows):
        """EXTENSION (agpt.h agpt_upload_emission): rows[i] = material i's agpt.emission(...), naming a texture of the last
        texture upload.  [] clears.  A texture upload clears the table."""
        rows = list(rows)
        for r in rows:
            if not isinstance(r, Emission):
                raise AgptError("upload_emission: every row must be an emission(...) row")
            if r.texture < -1 or not all(np.isfinite(f) and f >= 0 for f in r.factor):
                raise AgptError("upload_emission: need texture >= -1 and a finite factor >= 0")
        table = (Emission * max(len(rows), 1))(*rows)
        _check(core().agpt_upload_emission(self._h, table if rows else None, c_int(len(rows))))

    def set_camera(self, cam19):
        cam19 = np.ascontiguousarray(cam19, np.float32)
        assert cam19.size == 19
        _check(core().agpt_set_camera(self._h, _fptr(cam19)))

    def set_film(self, width, height):
        _check(core().agpt_set_film(self._h, c_int(width), c_int(height)))
        self.width, self.height = width, height

    def clear(self):
        _check(core().agpt_clear(self._h))

    def render(self, first_sample, num_samples, max_depth, depth_arg=0, flags=0, sample_stride=1):
        _check(core().agpt_render(self._h, c_int(first_sample), c_int(num_samples), c_int(sample_stride),
                                  c_int(max_depth), c_int(depth_arg), c_uint32(flags)))

    def read_accum(self, out=None):
        if out is None:
            out = np.empty((self.height, self.width, 4), np.float32)
        _check(core().agpt_read_accum(self._h, _fptr(out)))
        return out

    def write_accum(self, arr):
        arr = np.ascontiguousarray(arr, np.float32)
        assert arr.shape == (self.height, self.width, 4)
        _check(core().agpt_write_accum(self._h, _fptr(arr)))

    def write_accum_begin(self, arr):
        """agpt_write_accum_begin: the upload runs beside the render that follows; `arr` (C-contiguous float32, ideally
        page-locked: pinned_film) must stay untouched until the next call that touches the film returns."""
        assert arr.dtype == np.float32 and arr.flags["C_CONTIGUOUS"] and arr.shape == (self.height, self.width, 4)
        _check(core().agpt_write_accum_begin(self._h, _fptr(arr)))

    def accum_ptr(self):
        p = c_void_p()
        _check(core().agpt_accum_ptr_dev(self._h, byref(p)))
        return p.value

    def set_accum_dev(self, dev_ptr):
        _check(core().agpt_set_accum_dev(self._h, c_void_p(dev_ptr)))

    def resolve(self, samples):
        out = np.empty((self.height, self.width), np.uint32)
        _check(core().agpt_resolve(self._h, c_int(samples), out.ctypes.data_as(POINTER(c_uint32))))
        return out

    # ---- adaptive sampling (extension) -------------------------------------------------------------
    def set_moments(self, enable=True):
        """Per-pixel moments (sum of squares per channel, sample count) beside the film; off by default."""
        _check(core().agpt_set_moments(self._h, c_int(1 if enable else 0)))

    def read_moments(self, out=None):
        """float32 [H, W, 4] in the film's row order: .xyz = sum of c*c, .w = samples added."""
        if out is None:
            out = np.empty((self.height, self.width, 4), np.float32)
        _check(core().agpt_read_moments(self._h, _fptr(out)))
        return out

    def write_moments(self, arr):
        """Moments in read_moments' layout back to the device (resume an adaptive render along with write_accum)."""
        arr = np.ascontiguousarray(arr, np.float32)
        assert arr.shape == (self.height, self.width, 4)
        _check(core().agpt_write_moments(self._h, _fptr(arr)))

    def adaptive_select(self, params, want_pixels=True):
        """The convergence test over the film: (count, film pixel indices y*W + x of the selected pixels, or None)."""
        n = c_int(0)
        buf = np.empty(self.width * self.height, np.int32) if want_pixels else None
        _check(core().agpt_adaptive_select(self._h, byref(params), None if buf is None else buf.ctypes.data_as(POINTER(c_int32)), byref(n)))
        return n.value, (None if buf is None else buf[:n.value].copy())

    def render_adaptive(self, params, max_depth, depth_arg=0, flags=0):
        """A frame from scratch, adaptively: returns (rounds, camera paths)."""
        rounds = c_int(0); paths = c_int64(0)
        _check(core().agpt_render_adaptive(self._h, byref(params), c_int(max_depth), c_int(depth_arg), c_uint32(flags), byref(rounds), byref(paths)))
        return rounds.value, paths.value

    def resolve_counts(self):
        """agpt_resolve with each pixel's own sample count (moments .w)."""
        out = np.empty((self.height, self.width), np.uint32)
        _check(core().agpt_resolve_counts(self._h, out.ctypes.data_as(POINTER(c_uint32))))
        return out

    # ---- denoising (extension) ---------------------------------------------------------------------
    def render_guides(self, num_samples, flags=0):
        """First hits of the camera rays of samples [0, num_samples) of every pixel -> the context's guide buffers."""
        _check(core().agpt_render_guides(self._h, c_int(num_samples), c_uint32(flags)))

    def read_guides(self):
        """(albedo, normal_depth): float32 [H, W, 4] each, in the film's row order."""
        alb = np.empty((self.height, self.width, 4), np.float32)
        nd = np.empty((self.height, self.width, 4), np.float32)
        _check(core().agpt_read_guides(self._h, _fptr(alb), _fptr(nd)))
        return alb, nd

    def denoise(self, params):
        """The a-trous filter over the resident film, moments and guides: (float32 [H, W, 4] mean radiance, uint32 [H, W] packed
        pixels), both in the film's row order."""
        out = np.empty((self.height, self.width, 4), np.float32)
        rgb8 = np.empty((self.height, self.width), np.uint32)
        _check(core().agpt_denoise(self._h, byref(params), _fptr(out), rgb8.ctypes.data_as(POINTER(c_uint32))))
        return out, rgb8

    # ---- reprojection (extension) ------------------------------------------------------------------
    def reproject_film(self, params):
        """Carry the film and moments from the saved view into the current camera's (needs fresh guides), then save this view."""
        _check(core().agpt_reproject_film(self._h, byref(params)))

    def trace_primary(self, sample, flags=0):
        out = np.empty(self.width * self.height, HIT_DTYPE)
        _check(core().agpt_trace_primary(self._h, c_int(sample), c_uint32(flags), out.ctypes.data_as(c_void_p)))
        return out

    def trace_rays(self, rays7, any_hit=False, flags=0):
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        out = np.empty(len(rays7), HIT_DTYPE)
        _check(core().agpt_trace_rays(self._h, c_int64(len(rays7)), _fptr(rays7), c_int(1 if any_hit else 0),
                                      c_uint32(flags), out.ctypes.data_as(c_void_p)))
        return out

    def li_pixels(self, xs, ys, ss, max_depth, depth_arg=0, flags=0):
        xs = np.ascontiguousarray(xs, np.int32); ys = np.ascontiguousarray(ys, np.int32); ss = np.ascontiguousarray(ss, np.int32)
        out = np.empty((len(xs), 3), np.float32)
        ip = lambda a: a.ctypes.data_as(POINTER(c_int))
        _check(core().agpt_li_pixels(self._h, c_int(len(xs)), ip(xs), ip(ys), ip(ss), c_int(max_depth), c_int(depth_arg), c_uint32(flags), _fptr(out)))
        return out

    def li_rays(self, rays7, rng_states, max_depth, depth_arg=0, flags=0):
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        rng_states = np.ascontiguousarray(rng_states, np.uint32)
        out = np.empty((len(rays7), 3), np.float32)
        _check(core().agpt_li_rays(self._h, c_int(len(rays7)), _fptr(rays7), rng_states.ctypes.data_as(POINTER(c_uint32)),
                                   c_int(max_depth), c_int(depth_arg), c_uint32(flags), _fptr(out)))
        return out

    def stats(self):
        s = Stats()
        _check(core().agpt_get_stats(self._h, byref(s)))
        return s

    def reset_stats(self):
        _check(core().agpt_reset_stats(self._h))

    # ---- multi-process sharding: peers' accumulators through CUDA IPC ---------------------------
    def accum_ipc_handle(self):
        buf = ctypes.create_string_buffer(64)
        _check(core().agpt_accum_ipc_handle(self._h, buf))
        return buf.raw

    def open_peer_accums(self, rank, handles):
        """handles: list of 64-byte handles in rank order (own entry ignored)."""
        blob = b"".join(handles)
        assert len(blob) == 64 * len(handles)
        _check(core().agpt_open_peer_accums(self._h, c_int(rank), c_int(len(handles)), blob))

    def close_peer_accums(self):
        _check(core().agpt_close_peer_accums(self._h))

    def allreduce_accum_peers(self):
        _check(core().agpt_allreduce_accum_peers(self._h))

    def reduce_resolve_peers(self, samples, keep_sum=False):
        out = np.empty((self.height, self.width), np.uint32)
        _check(core().agpt_reduce_resolve_peers(self._h, c_int(samples), c_int(1 if keep_sum else 0), out.ctypes.data_as(POINTER(c_uint32))))
        return out

    def wave_stats(self, kind=0, max_waves=64):
        """Per-wave (= per-bounce) traversal counters of the COUNTERS renders since reset_stats: list of dicts."""
        rows = (c_uint64 * (8 * max_waves))()
        n = c_int(0)
        _check(core().agpt_get_wave_stats(self._h, c_int(kind), rows, c_int(max_waves), byref(n)))
        names = ("rays", "node_visits", "box_tests", "tri_tests", "analytic_tests", "warp_steps", "lane_steps")
        return [dict(zip(names, [int(rows[8 * w + k]) for k in range(7)])) for w in range(n.value)]

    def probe_bandwidth(self, nbytes, iters):
        g = c_float(0)
        _check(core().agpt_probe_bandwidth(self._h, ctypes.c_size_t(nbytes), c_int(iters), byref(g)))
        return g.value

    def debug_status(self):
        out = (c_uint64 * 4)()
        _check(core().agpt_debug_status(self._h, out))
        return dict(failed=out[0], first_code=out[1], first_value=out[2], checks=out[3])

    def scene_bytes(self):
        b = c_uint64(0)
        _check(core().agpt_scene_bytes(self._h, byref(b)))
        return b.value

    # ---- probes -------------------------------------------------------------------------
    def probe_bounds(self, boxes6, rays7):
        boxes6 = np.ascontiguousarray(boxes6, np.float32).reshape(-1, 6)
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        n = len(boxes6)
        hit = np.empty(n, np.int32); t = np.empty(n, np.float32)
        _check(core().agpt_probe_bounds(self._h, c_int(n), _fptr(boxes6), _fptr(rays7), hit.ctypes.data_as(POINTER(c_int)), _fptr(t)))
        return hit, t

    def probe_bsdf(self, material, in14, skip_specular):
        in14 = np.ascontiguousarray(in14, np.float32).reshape(-1, 14)
        out = np.empty((len(in14), 12), np.float32)
        _check(core().agpt_probe_bsdf(self._h, c_int(len(in14)), byref(material), _fptr(in14), c_int(1 if skip_specular else 0), _fptr(out)))
        return out

    def probe_sphere_sample(self, in9):
        in9 = np.ascontiguousarray(in9, np.float32).reshape(-1, 9)
        out = np.empty((len(in9), 8), np.float32)
        _check(core().agpt_probe_sphere_sample(self._h, c_int(len(in9)), _fptr(in9), _fptr(out)))
        return out

    def probe_light_sample(self, light, in8):
        """Extension: Sample_Li / Pdf_Li of resident light `light` (an area light with LIGHT_SAMPLE_SHAPE on a plane or mesh).
        in8 rows: ref point, u (2), query direction; out rows: sampled point, its pdf, Pdf_Li(query direction), light normal."""
        in8 = np.ascontiguousarray(in8, np.float32).reshape(-1, 8)
        out = np.empty((len(in8), 8), np.float32)
        _check(core().agpt_probe_light_sample(self._h, c_int(light), c_int(len(in8)), _fptr(in8), _fptr(out)))
        return out

    def probe_material_maps(self, rays7):
        """EXTENSION (agpt.h agpt_probe_material_maps): per ray, 32 floats: prim (-1 miss), u, v, ng, ns, ss, ts, T, B, roughness,
        metallic, lobes, diffuse_r, spec_r0 of the closest hit as the maps shade kernel builds them."""
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        out = np.zeros((len(rays7), 32), np.float32)
        _check(core().agpt_probe_material_maps(self._h, c_int(len(rays7)), _fptr(rays7), _fptr(out)))
        return out

    def probe_stream(self, pixel_index, sample, k):
        out = np.empty(k, np.float32)
        _check(core().agpt_probe_stream(self._h, c_uint32(pixel_index), c_uint32(sample), c_int(k), _fptr(out)))
        return out


class Group:
    """Contexts of this process, one per GPU, that split a render by sample index (SURVEY 8e)."""

    def __init__(self, contexts):
        self.contexts = list(contexts)
        self._arr = (c_void_p * len(self.contexts))(*[c.handle for c in self.contexts])

    def __len__(self):
        return len(self.contexts)

    def render(self, first_sample, num_samples, max_depth, depth_arg=0, flags=0):
        _check(core().agpt_render_multi(self._arr, c_int(len(self)), c_int(first_sample), c_int(num_samples), c_int(max_depth), c_int(depth_arg), c_uint32(flags)))

    def reduce(self, root=-1):
        """Sum of the accumulators, in rank order: into every context (root = -1) or into contexts[root] only."""
        _check(core().agpt_reduce_accum(self._arr, c_int(len(self)), c_int(root)))

    def reduce_resolve(self, samples, keep_sum=False):
        c0 = self.contexts[0]
        out = np.empty((c0.height, c0.width), np.uint32)
        _check(core().agpt_reduce_resolve(self._arr, c_int(len(self)), c_int(samples), c_int(1 if keep_sum else 0), out.ctypes.data_as(POINTER(c_uint32))))
        return out


def pinned_film(width, height):
    """float32 [H, W, 4] numpy view over page-locked host memory (agpt_host_alloc); keep the
    returned owner object alive as long as the array is used."""
    nbytes = width * height * 16
    p = c_void_p()
    _check(core().agpt_host_alloc(ctypes.c_size_t(nbytes), byref(p)))
    buf = (c_float * (width * height * 4)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=np.float32).reshape(height, width, 4)
    arr[:] = 0

    class _Owner:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            try:
                core().agpt_host_free(c_void_p(self.ptr))
            except Exception:
                pass
    return arr, _Owner(p.value)


def make_material(mtype, color, roughness=0.0, metallic=0.0):
    m = Material()
    col = (c_float * 3)(*[float(v) for v in color])
    _check(host().agpt_host_make_material(c_int(mtype), col, c_float(roughness), c_float(metallic), byref(m)), host_side=True)
    return m


def set_build_options(threads=0, cache_dir=None):
    """BVH builder threads (>= 1) and cache directory ('' = off) of the host mirror."""
    _check(host().agpt_host_set_build_options(c_int(threads), None if cache_dir is None else str(cache_dir).encode()), host_side=True)


def get_build_options():
    t = c_int()
    buf = ctypes.create_string_buffer(4096)
    _check(host().agpt_host_get_build_options(byref(t), buf, c_int(4096)), host_side=True)
    return t.value, buf.value.decode()


def config_defaults(config):
    out = (c_int * 5)()
    name = c_char_p()
    _check(host().agpt_host_config_defaults(c_int(config), out, byref(name)), host_side=True)
    return dict(width=out[0], height=out[1], spp=out[2], max_depth=out[3], depth_arg=out[4], name=name.value.decode())


class HostScene:
    """A BASELINE.json configuration built through the host mirror of the reference API."""

    def __init__(self, config, level=0):
        self._h = c_void_p()
        _check(host().agpt_host_scene_create(c_int(config), c_int(level), byref(self._h)), host_side=True)
        self.config, self.level = config, level

    def close(self):
        if self._h:
            host().agpt_host_scene_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def counts(self):
        c = (c_int64 * 4)(); b = c_uint64(0)
        _check(host().agpt_host_scene_counts(self._h, c, byref(b)), host_side=True)
        return dict(prims=c[0], lights=c[1], tris=c[2], nodes=c[3], bytes=b.value)

    def upload(self, ctx):
        _check(host().agpt_host_scene_upload(self._h, ctx.handle), host_side=True)

    def camera(self):
        out = np.empty(19, np.float32)
        _check(host().agpt_host_camera_export(self._h, _fptr(out)), host_side=True)
        return out

    def tables(self):
        """agpt_scene_tables view (opaque bytes) of the flattened scene, valid while the scene lives."""
        buf = ctypes.create_string_buffer(512)       # sizeof(agpt_scene_tables) = 264
        _check(host().agpt_host_scene_tables(self._h, buf), host_side=True)
        return buf

    def prim_info(self, prim):
        kind = c_int(); counts = (c_int * 5)(); hm = c_int(); il = c_int()
        _check(host().agpt_host_prim_info(self._h, c_int(prim), byref(kind), counts, byref(hm), byref(il)), host_side=True)
        return dict(kind=kind.value, nodes=counts[0], tris=counts[1], has_normals=bool(counts[3]), has_uvs=bool(counts[4]),
                    has_material=bool(hm.value), is_light=bool(il.value))

    def bvh(self, prim):
        info = self.prim_info(prim)
        nodes = np.zeros((info["nodes"], 8), np.uint32)
        order = np.zeros(info["tris"], np.int32)
        n = _check(host().agpt_host_bvh_export(self._h, c_int(prim), nodes.ctypes.data_as(c_void_p), order.ctypes.data_as(POINTER(c_int))), host_side=True)
        return nodes[:n], order

    def mesh_verts(self, prim):
        info = self.prim_info(prim)
        v = np.zeros((info["tris"], 9), np.float32)
        _check(host().agpt_host_mesh_export(self._h, c_int(prim), _fptr(v)), host_side=True)
        return v

    def alpha_masks(self):
        """EXTENSION: the flattened scene's alpha-mask rows (agpt_host_scene_alpha_masks), one per material, or [] without masks."""
        p = POINTER(AlphaMask)(); n = c_int(0)
        _check(host().agpt_host_scene_alpha_masks(self._h, byref(p), byref(n)), host_side=True)
        return [AlphaMask(p[i].texture, p[i].channel, p[i].cutoff, 0) for i in range(n.value)]

    def emission(self):
        """EXTENSION: the flattened scene's emission rows (agpt_host_scene_emission), one per material, or [] when none emits."""
        p = POINTER(Emission)(); n = c_int(0)
        _check(host().agpt_host_scene_emission(self._h, byref(p), byref(n)), host_side=True)
        return [Emission(p[i].texture, (c_float * 3)(*p[i].factor)) for i in range(n.value)]

    def material(self, prim):
        out = np.zeros(20, np.float32)
        _check(host().agpt_host_material_export(self._h, c_int(prim), _fptr(out)), host_side=True)
        return out


class HostTracer:
    """CudaPathTracer: the reference-facing integrator object (host buffers in and out)."""

    def __init__(self, max_depth=5, device=0, devices=None):
        self._h = c_void_p()
        if devices is None:
            _check(host().agpt_host_tracer_create(c_int(max_depth), c_int(device), byref(self._h)), host_side=True)
        else:
            arr = (c_int * len(devices))(*devices)
            _check(host().agpt_host_tracer_create_multi(c_int(max_depth), arr, c_int(len(devices)), byref(self._h)), host_side=True)

    def close(self):
        if self._h:
            host().agpt_host_tracer_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def render(self, scene, width, height, accum, first_sample, num_samples, depth_arg=0, flags=0, reupload=False):
        assert accum.dtype == np.float32 and accum.shape == (height, width, 4) and accum.flags.c_contiguous
        _check(host().agpt_host_tracer_render(self._h, scene.handle, c_int(width), c_int(height), _fptr(accum), c_int(first_sample),
                                              c_int(num_samples), c_int(depth_arg), c_uint32(flags), c_int(1 if reupload else 0)), host_side=True)
        return accum

    def stats(self, reset=False):
        """agpt_stats of the tracer's first context (CudaPathTracer::Context())."""
        ctx = c_void_p()
        _check(host().agpt_host_tracer_ctx(self._h, byref(ctx)), host_side=True)
        s = Stats()
        _check(core().agpt_get_stats(ctx, byref(s)))
        if reset:
            _check(core().agpt_reset_stats(ctx))
        return s

    def render_resolve(self, scene, width, height, accum, samples_so_far, first_sample, num_samples, depth_arg=0, flags=0):
        """RenderAndResolve: returns the packed 0x00RRGGBB image of the film after these samples."""
        assert accum.dtype == np.float32 and accum.shape == (height, width, 4) and accum.flags.c_contiguous
        out = np.empty((height, width), np.uint32)
        _check(host().agpt_host_tracer_render_resolve(self._h, scene.handle, c_int(width), c_int(height), _fptr(accum), c_int(samples_so_far),
                                                      c_int(first_sample), c_int(num_samples), c_int(depth_arg), c_uint32(flags),
                                                      out.ctypes.data_as(POINTER(c_uint32))), host_side=True)
        return out

    def render_adaptive(self, scene, width, height, accum, params, depth_arg=0, flags=0):
        """CudaPathTracer::RenderAdaptive: the film replaces `accum`; returns the per-pixel sample counts [H, W] (row 0 = top)."""
        assert accum.dtype == np.float32 and accum.shape == (height, width, 4) and accum.flags.c_contiguous
        counts = np.empty((height, width), np.int32)
        _check(host().agpt_host_tracer_render_adaptive(self._h, scene.handle, c_int(width), c_int(height), _fptr(accum), byref(params),
                                                       c_int(depth_arg), c_uint32(flags), counts.ctypes.data_as(POINTER(c_int32))), host_side=True)
        return counts

    def render_adaptive_denoised(self, scene, width, height, accum, params, denoise, guide_samples, depth_arg=0, flags=0):
        """CudaPathTracer::RenderAdaptiveDenoised: the film replaces `accum`; returns (counts [H, W] with row 0 = top, denoised
        float32 [H, W, 4] and packed uint32 [H, W], both in the film's row order)."""
        assert accum.dtype == np.float32 and accum.shape == (height, width, 4) and accum.flags.c_contiguous
        counts = np.empty((height, width), np.int32)
        out = np.empty((height, width, 4), np.float32)
        rgb8 = np.empty((height, width), np.uint32)
        _check(host().agpt_host_tracer_render_adaptive_denoised(self._h, scene.handle, c_int(width), c_int(height), _fptr(accum), byref(params),
                                                                byref(denoise), c_int(guide_samples), c_int(depth_arg), c_uint32(flags),
                                                                counts.ctypes.data_as(POINTER(c_int32)), _fptr(out),
                                                                rgb8.ctypes.data_as(POINTER(c_uint32))), host_side=True)
        return counts, out, rgb8

    def render_temporal(self, scene, width, height, accum, first_sample, num_samples, reproject, denoise, guide_samples, camera=None,
                        depth_arg=0, flags=0):
        """CudaPathTracer::RenderTemporal with `camera` (19 floats of agpt_camera, None: the scene's): the film replaces `accum`;
        returns (denoised float32 [H, W, 4], packed uint32 [H, W]), both in the film's row order."""
        assert accum.dtype == np.float32 and accum.shape == (height, width, 4) and accum.flags.c_contiguous
        out = np.empty((height, width, 4), np.float32)
        rgb8 = np.empty((height, width), np.uint32)
        cam = None if camera is None else np.ascontiguousarray(camera, np.float32)
        assert cam is None or cam.size == 19
        _check(host().agpt_host_tracer_render_temporal(self._h, scene.handle, None if cam is None else cam.ctypes.data_as(c_void_p), c_int(width),
                                                       c_int(height), _fptr(accum), c_int(first_sample), c_int(num_samples), byref(reproject),
                                                       byref(denoise), c_int(guide_samples), c_int(depth_arg), c_uint32(flags), _fptr(out),
                                                       rgb8.ctypes.data_as(POINTER(c_uint32))), host_side=True)
        return out, rgb8

    def li(self, scene, origin, direction, depth_arg=0):
        o = (c_float * 3)(*origin); d = (c_float * 3)(*direction); out = (c_float * 3)()
        _check(host().agpt_host_tracer_li(self._h, scene.handle, o, d, c_int(depth_arg), out), host_side=True)
        return np.array(list(out), np.float32)
