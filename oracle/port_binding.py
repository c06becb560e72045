"""ctypes binding over oracle/libagpt_oracle.so (the plain-C++ restatement) -- TEST INFRASTRUCTURE."""
import ctypes
import os
from ctypes import POINTER, c_float, c_int, c_longlong, c_uint, c_ulonglong, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libagpt_oracle.so")
HIT_DTYPE = np.dtype([("found", np.uint32), ("prim", np.int32), ("tri", np.int32), ("t", np.float32)])
_lib = None


def available():
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError(f"{LIB_PATH} missing: run `make -C oracle port`")
        L = ctypes.CDLL(LIB_PATH)
        L.agpt_oracle_scene_create.restype = c_void_p
        L.agpt_oracle_render.restype = c_longlong
        L.agpt_oracle_primary_hits.restype = c_longlong
        _lib = L
    return _lib


def _fp(a):
    return a.ctypes.data_as(POINTER(c_float))


class _Tables(ctypes.Structure):       # agpt_oracle_tables (= agpt_scene_tables of include/agpt_host.h)
    _fields_ = [("prims", c_void_p), ("n_prims", c_int), ("spheres", c_void_p), ("n_spheres", c_int), ("planes", c_void_p), ("n_planes", c_int),
                ("meshes", c_void_p), ("n_meshes", c_int), ("materials", c_void_p), ("n_materials", c_int), ("lights", c_void_p), ("n_lights", c_int),
                ("camera", c_float * 19), ("env_w", c_int), ("env_h", c_int), ("env_rgb", c_void_p), ("env_func", c_void_p), ("env_cdf", c_void_p),
                ("env_func_int", c_float), ("instances", c_void_p), ("n_instances", c_int)]


class PortScene:
    """The restatement fed with the flattened tables of a host-mirror scene (HostScene.tables()),
    or with hand-built tables (PortScene.from_tables)."""

    def __init__(self, host_scene=None, tables=None, keep=None):
        self._keep = host_scene if host_scene is not None else keep       # the tables borrow this memory
        self._h = c_void_p(lib().agpt_oracle_scene_create(host_scene.tables() if host_scene is not None else ctypes.byref(tables)))

    @classmethod
    def from_tables(cls, prims, meshes=(), spheres=None, planes=None, materials=(), lights=None, camera=None, instances=None):
        """prims / spheres / planes / lights: structured numpy arrays in the layouts of include/agpt.h;
        meshes: objects with .desc() -> agpt_mesh_desc (binding.RawMesh); materials: list of agpt_material."""
        t = _Tables()
        keep = [prims, meshes, spheres, planes, materials, lights]
        def put(name, count, arr):
            setattr(t, name, arr.ctypes.data if arr is not None and len(arr) else None)
            setattr(t, count, 0 if arr is None else len(arr))
        put("prims", "n_prims", prims); put("spheres", "n_spheres", spheres); put("planes", "n_planes", planes); put("lights", "n_lights", lights)
        put("instances", "n_instances", instances); keep.append(instances)
        if len(meshes):
            descs = (type(meshes[0].desc()) * len(meshes))(*[m.desc() for m in meshes])
            keep.append(descs)
            t.meshes = ctypes.addressof(descs); t.n_meshes = len(meshes)
        if len(materials):
            mats = (type(materials[0]) * len(materials))(*materials)
            keep.append(mats)
            t.materials = ctypes.addressof(mats); t.n_materials = len(materials)
        if camera is not None:
            t.camera = (c_float * 19)(*[float(v) for v in camera])
        return cls(tables=t, keep=keep)

    def set_rr_by_bounce(self, on=True):
        """EXTENSION (not reference behaviour): Russian roulette keyed on the bounce index, bounces > 3."""
        lib().agpt_oracle_scene_set_rr_by_bounce(self._h, c_int(1 if on else 0))

    def trace_rays(self, rays7, any_hit=False):
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        hits = np.zeros(len(rays7), HIT_DTYPE)
        st = (c_ulonglong * 3)()
        lib().agpt_oracle_trace_rays(self._h, c_longlong(len(rays7)), _fp(rays7), c_int(1 if any_hit else 0), hits.ctypes.data_as(c_void_p), st)
        return hits, dict(interior=st[0], boxes=st[1], tris=st[2])

    def close(self):
        if self._h:
            lib().agpt_oracle_scene_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def render(self, W, H, s0, ns, max_depth, depth_arg=0, threads=0, crop=None, out=None, sample_stride=1):
        if out is None:
            out = np.zeros((H, W, 4), np.float32)
        x0, y0, x1, y1 = crop if crop else (0, 0, W, H)
        threads = threads or os.cpu_count() or 1
        cnt = (c_ulonglong * 6)()
        n = lib().agpt_oracle_render(self._h, c_int(W), c_int(H), c_int(x0), c_int(y0), c_int(x1), c_int(y1), c_int(s0), c_int(ns),
                                     c_int(sample_stride), c_int(max_depth), c_int(depth_arg), c_int(threads), _fp(out), cnt)
        names = ["rays_closest", "rays_any", "interior", "boxes", "tris", "analytic"]
        return out, dict(zip(names, list(cnt)), paths=n)

    def primary_hits(self, W, H, sample, threads=0, want_counts=False):
        hits = np.zeros(W * H, HIT_DTYPE)
        st = (c_ulonglong * 3)()
        lib().agpt_oracle_primary_hits(self._h, c_int(W), c_int(H), c_int(sample), c_int(threads or os.cpu_count() or 1), hits.ctypes.data_as(c_void_p), st)
        return (hits, dict(interior=st[0], boxes=st[1], tris=st[2])) if want_counts else hits

    def li_pixels(self, W, H, xs, ys, ss, max_depth, depth_arg=0):
        xs = np.ascontiguousarray(xs, np.int32); ys = np.ascontiguousarray(ys, np.int32); ss = np.ascontiguousarray(ss, np.int32)
        out = np.zeros((len(xs), 3), np.float32); draws = np.zeros(len(xs), np.int32)
        ip = lambda a: a.ctypes.data_as(POINTER(c_int))
        lib().agpt_oracle_li_pixels(self._h, c_int(W), c_int(H), c_int(len(xs)), ip(xs), ip(ys), ip(ss), c_int(max_depth), c_int(depth_arg), _fp(out), ip(draws))
        return out, draws


def probe_bsdf(material, in14, skip_specular):
    """BSDF::f / Pdf / Sample_f of the restatement for an agpt_material record (ctypes struct)."""
    in14 = np.ascontiguousarray(in14, np.float32).reshape(-1, 14)
    out = np.zeros((len(in14), 12), np.float32)
    lib().agpt_oracle_probe_bsdf(c_int(len(in14)), ctypes.byref(material), _fp(in14), c_int(1 if skip_specular else 0), _fp(out))
    return out


def probe_stream(pixel, sample, k):
    out = np.zeros(k, np.float32)
    lib().agpt_oracle_probe_stream(c_uint(pixel), c_uint(sample), c_int(k), _fp(out))
    return out
