"""ctypes binding over oracle/libagpt_shape_oracle.so -- TEST INFRASTRUCTURE.

EXTENSION: the CPU statement of sampled plane and mesh area lights (include/agpt.h AGPT_LIGHT_SAMPLE_SHAPE), built on the
oracle (oracle/agpt_shape_oracle.cpp).  ShapeScene takes the same tables as port_binding.PortScene and renders, traces and
probes with the extension; with no light flagged it renders what PortScene renders."""
import ctypes
import os
from ctypes import POINTER, c_float, c_int, c_longlong, c_ulonglong, c_void_p

import numpy as np

from .port_binding import HIT_DTYPE, _Tables  # noqa: F401  (_Tables: the agpt_oracle_tables layout, re-exported for tests)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libagpt_shape_oracle.so")
_lib = None


def available():
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError(f"{LIB_PATH} missing: run __graft_entry__.build()")
        L = ctypes.CDLL(LIB_PATH)
        L.agpt_shape_oracle_scene_create.restype = c_void_p
        L.agpt_shape_oracle_render.restype = c_longlong
        _lib = L
    return _lib


def _fp(a):
    return a.ctypes.data_as(POINTER(c_float))


class ShapeScene:
    """The statement fed with the flattened tables of a host-mirror scene (HostScene.tables()), or with hand-built tables
    (ShapeScene.from_tables, the arguments of port_binding.PortScene.from_tables)."""

    def __init__(self, host_scene=None, tables=None, keep=None):
        self._keep = host_scene if host_scene is not None else keep       # the tables borrow this memory
        self._h = c_void_p(lib().agpt_shape_oracle_scene_create(host_scene.tables() if host_scene is not None else ctypes.byref(tables)))

    @classmethod
    def from_tables(cls, prims, meshes=(), spheres=None, planes=None, materials=(), lights=None, camera=None, instances=None):
        t = _Tables()
        keep = [prims, meshes, spheres, planes, materials, lights, instances]
        def put(name, count, arr):
            setattr(t, name, arr.ctypes.data if arr is not None and len(arr) else None)
            setattr(t, count, 0 if arr is None else len(arr))
        put("prims", "n_prims", prims); put("spheres", "n_spheres", spheres); put("planes", "n_planes", planes); put("lights", "n_lights", lights)
        put("instances", "n_instances", instances)
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

    def close(self):
        if self._h:
            lib().agpt_shape_oracle_scene_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_rr_by_bounce(self, on=True):
        lib().agpt_shape_oracle_scene_set_rr_by_bounce(self._h, c_int(1 if on else 0))

    def trace_rays(self, rays7, any_hit=False):
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        hits = np.zeros(len(rays7), HIT_DTYPE)
        st = (c_ulonglong * 3)()
        lib().agpt_shape_oracle_trace_rays(self._h, c_longlong(len(rays7)), _fp(rays7), c_int(1 if any_hit else 0), hits.ctypes.data_as(c_void_p), st)
        return hits, dict(interior=st[0], boxes=st[1], tris=st[2])

    def render(self, W, H, s0, ns, max_depth, depth_arg=0, threads=0, crop=None, out=None, sample_stride=1):
        if out is None:
            out = np.zeros((H, W, 4), np.float32)
        x0, y0, x1, y1 = crop if crop else (0, 0, W, H)
        threads = threads or os.cpu_count() or 1
        cnt = (c_ulonglong * 6)()
        n = lib().agpt_shape_oracle_render(self._h, c_int(W), c_int(H), c_int(x0), c_int(y0), c_int(x1), c_int(y1), c_int(s0), c_int(ns),
                                           c_int(sample_stride), c_int(max_depth), c_int(depth_arg), c_int(threads), _fp(out), cnt)
        names = ["rays_closest", "rays_any", "interior", "boxes", "tris", "analytic"]
        return out, dict(zip(names, list(cnt)), paths=n)

    def li_pixels(self, W, H, xs, ys, ss, max_depth, depth_arg=0):
        xs = np.ascontiguousarray(xs, np.int32); ys = np.ascontiguousarray(ys, np.int32); ss = np.ascontiguousarray(ss, np.int32)
        out = np.zeros((len(xs), 3), np.float32); draws = np.zeros(len(xs), np.int32)
        ip = lambda a: a.ctypes.data_as(POINTER(c_int))
        lib().agpt_shape_oracle_li_pixels(self._h, c_int(W), c_int(H), c_int(len(xs)), ip(xs), ip(ys), ip(ss), c_int(max_depth), c_int(depth_arg),
                                          _fp(out), ip(draws))
        return out, draws

    def probe_light_sample(self, light, in8):
        """agpt_probe_light_sample's contract: in8 rows ref point, u (2), query direction; out rows sampled point, its pdf,
        Pdf_Li(query direction), light normal."""
        in8 = np.ascontiguousarray(in8, np.float32).reshape(-1, 8)
        out = np.zeros((len(in8), 8), np.float32)
        lib().agpt_shape_oracle_probe_light_sample(self._h, c_int(light), c_int(len(in8)), _fp(in8), _fp(out))
        return out
