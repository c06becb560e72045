"""ctypes binding over statements/libagpt_material_maps_oracle.so -- TEST INFRASTRUCTURE.

EXTENSION: the CPU statement of roughness-metallic and normal maps on Disney materials (include/agpt.h
agpt_upload_material_textures), built on the texture statement (statements/agpt_material_maps_oracle.cpp).  MapsScene takes
the tables of a host-mirror scene (HostScene.tables()), map bindings included; set_textures replaces them."""
import ctypes
import os
from ctypes import c_int, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libagpt_material_maps_oracle.so")
_lib = None

MAT_DTYPE = np.dtype([("type", np.int32), ("lobes", np.uint32), ("roughness", np.float32), ("metallic", np.float32), ("diffuse_r", np.float32, 3),
                      ("eta", np.float32), ("spec_r0", np.float32, 3), ("alpha_x", np.float32), ("mirror_r", np.float32, 3), ("alpha_y", np.float32)])


class _Texture(ctypes.Structure):      # agpt_texture
    _fields_ = [("width", c_int), ("height", c_int), ("rgb", ctypes.POINTER(ctypes.c_float))]


def available():
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError(f"{LIB_PATH} missing: run __graft_entry__.build()")
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.agpt_maps_oracle_create.restype = c_void_p
    return _lib


def _p(a):
    return a.ctypes.data_as(c_void_p)


def frame(N, T, B, texel, scale):
    """The normal-map rule on a surface with shading normal N and shading dpdu T: (sn, sdpdu, changed) per row."""
    rows = np.ascontiguousarray(np.concatenate([np.reshape(x, (-1, 3)) for x in (N, T, B, texel)], axis=1), np.float32)
    scale = np.ascontiguousarray(np.broadcast_to(np.float32(scale), (len(rows),)), np.float32)
    out = np.zeros((len(rows), 7), np.float32)
    lib().agpt_maps_oracle_frame(c_int(len(rows)), _p(rows), _p(scale), _p(out))
    return out[:, 0:3], out[:, 3:6], out[:, 6] != 0


def material(rec, C, c):
    """The record DisneyMaterial's arithmetic derives from `rec` (a MAT_DTYPE row) with base colour C and texel c."""
    rec = np.ascontiguousarray(np.array(rec, MAT_DTYPE).reshape(1))
    out = np.zeros(1, MAT_DTYPE)
    C = np.ascontiguousarray(C, np.float32); c = np.ascontiguousarray(c, np.float32)
    lib().agpt_maps_oracle_material(_p(rec), _p(C), _p(c), _p(out))
    return out[0]


class MapsScene:
    def __init__(self, host_scene, rr_by_bounce=False):
        self._keep = host_scene                 # the tables borrow its memory
        self._h = c_void_p(lib().agpt_maps_oracle_create(host_scene.tables()))
        lib().agpt_maps_oracle_set_rr_by_bounce(self._h, c_int(1 if rr_by_bounce else 0))

    def set_textures(self, images, bindings):
        """The arguments of Context.upload_material_textures: images (H, W, 3) and agpt.material_textures(...) rows."""
        self._imgs = [np.ascontiguousarray(a, np.float32) for a in images]
        rows = (_Texture * max(len(self._imgs), 1))(*[_Texture(a.shape[1], a.shape[0], a.ctypes.data_as(ctypes.POINTER(ctypes.c_float)))
                                                      for a in self._imgs])
        size = 28                           # sizeof(agpt_material_textures)
        self._table = (ctypes.c_byte * (size * max(len(bindings), 1)))()
        for i, b in enumerate(bindings):
            assert ctypes.sizeof(b) == size
            ctypes.memmove(ctypes.addressof(self._table) + size * i, ctypes.addressof(b), size)
        self._rows = rows
        lib().agpt_maps_oracle_set_textures(self._h, rows, c_int(len(self._imgs)), self._table, c_int(len(bindings)))

    def close(self):
        if self._h:
            lib().agpt_maps_oracle_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def render(self, W, H, first, n, max_depth, depth_arg, threads=0, counters=False):
        """H x W float4 film (film row order) of samples [first, first + n), as agpt_render adds them; with counters=True also the
        statement's ray counts {rays_closest, rays_any, interior, boxes, tris, analytic}."""
        out = np.zeros((H, W, 4), np.float32)
        cnt = (ctypes.c_ulonglong * 6)()
        lib().agpt_maps_oracle_render(self._h, c_int(W), c_int(H), c_int(first), c_int(n), c_int(max_depth), c_int(depth_arg),
                                      c_int(threads or os.cpu_count() or 1), _p(out), cnt)
        if not counters:
            return out
        return out, dict(zip(["rays_closest", "rays_any", "interior", "boxes", "tris", "analytic"], list(cnt)))

    def li_pixels(self, W, H, xs, ys, ss, max_depth, depth_arg):
        xs, ys, ss = (np.ascontiguousarray(a, np.int32) for a in (xs, ys, ss))
        out = np.zeros((len(xs), 3), np.float32)
        lib().agpt_maps_oracle_li_pixels(self._h, c_int(W), c_int(H), c_int(len(xs)), _p(xs), _p(ys), _p(ss), c_int(max_depth), c_int(depth_arg), _p(out))
        return out

    def guides(self, W, H, num_samples, threads=0):
        alb = np.zeros((H, W, 4), np.float32)
        nd = np.zeros((H, W, 4), np.float32)
        lib().agpt_maps_oracle_guides(self._h, c_int(W), c_int(H), c_int(num_samples), c_int(threads or os.cpu_count() or 1), _p(alb), _p(nd))
        return alb, nd

    def hit_rows(self, rays7):
        """Per ray, 32 floats: prim (-1 miss), u, v, ng, sn, ss, ts (BSDF frame), T, B, roughness, metallic, lobes, diffuse_r, spec_r0."""
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        out = np.zeros((len(rays7), 32), np.float32)
        lib().agpt_maps_oracle_hit_rows(self._h, c_int(len(rays7)), _p(rays7), _p(out))
        return out

    def hit_triangle(self, rays7):
        """Per ray, 15 floats: the world-space vertices and uvs of the triangle hit (NaN: a miss, a sphere or a plane)."""
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        out = np.zeros((len(rays7), 15), np.float32)
        lib().agpt_maps_oracle_hit_triangle(self._h, c_int(len(rays7)), _p(rays7), _p(out))
        return out
