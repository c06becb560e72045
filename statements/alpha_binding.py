"""ctypes binding over statements/libagpt_alpha_oracle.so -- TEST INFRASTRUCTURE.

EXTENSION: the CPU statement of alpha-masked cutout geometry (include/agpt.h agpt_upload_alpha_masks), built on the maps
statement (statements/agpt_alpha_oracle.cpp).  AlphaScene takes the tables and the alpha masks of a host-mirror scene
(HostScene.tables(), HostScene.alpha_masks()), or hand-built tables (AlphaScene.from_tables); set_textures and set_masks replace
them as the device calls do."""
import ctypes
import os
from ctypes import c_float, c_int, c_longlong, c_void_p

import numpy as np

from oracle import port_binding

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libagpt_alpha_oracle.so")
_lib = None

HIT_DTYPE = np.dtype([("found", np.uint32), ("prim", np.int32), ("tri", np.int32), ("t", np.float32)])


class _Texture(ctypes.Structure):      # agpt_texture
    _fields_ = [("width", c_int), ("height", c_int), ("rgb", ctypes.POINTER(ctypes.c_float))]


class _Tables(port_binding._Tables):   # agpt_scene_tables of include/agpt_host.h: the oracle's tables, then the image tables
    _fields_ = [("textures", c_void_p), ("material_texture", c_void_p), ("n_textures", c_int), ("n_material_texture", c_int),
                ("material_textures", c_void_p), ("n_material_textures", c_int)]


class _Keep:                          # what hand-built tables borrow, with the tables() of a host-mirror scene
    def __init__(self, tables, keep):
        self._t, self._keep = tables, keep

    def tables(self):
        return ctypes.byref(self._t)


def available():
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError(f"{LIB_PATH} missing: run __graft_entry__.build()")
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.agpt_alpha_oracle_create.restype = c_void_p
    return _lib


def _p(a):
    return a.ctypes.data_as(c_void_p)


def _table(rows, size):
    """A packed C array of ctypes structures (agpt_alpha_mask: 16 bytes, agpt_material_textures: 28)."""
    buf = (ctypes.c_byte * (size * max(len(rows), 1)))()
    for i, b in enumerate(rows):
        assert ctypes.sizeof(b) == size
        ctypes.memmove(ctypes.addressof(buf) + size * i, ctypes.addressof(b), size)
    return buf


def _counters(cnt):
    return dict(zip(["rays_closest", "rays_any", "interior", "boxes", "tris", "analytic"], list(cnt)))


def lookup_channel(image, channel, uv):
    """Channel `channel` of the bilinear, repeat-wrapped lookup of image (H, W, 3) at each uv row."""
    img = np.ascontiguousarray(image, np.float32)
    uv = np.ascontiguousarray(uv, np.float32).reshape(-1, 2)
    out = np.zeros(len(uv), np.float32)
    lib().agpt_alpha_oracle_lookup_channel(c_int(img.shape[1]), c_int(img.shape[0]), _p(img), c_int(channel), c_int(len(uv)), _p(uv), _p(out))
    return out


class AlphaScene:
    def __init__(self, host_scene, masks=None, rr_by_bounce=False):
        self._keep = host_scene                 # the tables borrow its memory
        masks = host_scene.alpha_masks() if masks is None else list(masks)
        self._masks = _table(masks, 16)
        self._h = c_void_p(lib().agpt_alpha_oracle_create(host_scene.tables(), self._masks if masks else None, c_int(len(masks))))
        lib().agpt_alpha_oracle_set_rr_by_bounce(self._h, c_int(1 if rr_by_bounce else 0))

    @classmethod
    def from_tables(cls, prims, meshes=(), spheres=None, planes=None, materials=(), lights=None, instances=None, images=(), bindings=(),
                    masks=(), camera=None):
        """Hand-built tables in the layouts of include/agpt.h, as the raw C ABI takes them: prims / spheres / planes / lights /
        instances structured numpy arrays, meshes binding.RawMesh objects, materials agpt_material rows; images, bindings and masks
        the arguments of Context.upload_material_textures and Context.upload_alpha_masks."""
        t = _Tables()
        keep = [prims, spheres, planes, lights, instances]
        for name, arr in (("prims", prims), ("spheres", spheres), ("planes", planes), ("lights", lights), ("instances", instances)):
            if arr is not None and len(arr):
                arr = np.ascontiguousarray(arr)
                keep.append(arr)
                setattr(t, name, arr.ctypes.data); setattr(t, "n_" + name, len(arr))
        if len(meshes):
            descs = (type(meshes[0].desc()) * len(meshes))(*[m.desc() for m in meshes])
            keep += [descs, meshes]
            t.meshes = ctypes.addressof(descs); t.n_meshes = len(meshes)
        if len(materials):
            mats = (type(materials[0]) * len(materials))(*materials)
            keep.append(mats)
            t.materials = ctypes.addressof(mats); t.n_materials = len(materials)
        if camera is not None:
            t.camera = (c_float * 19)(*[float(v) for v in camera])
        imgs = [np.ascontiguousarray(a, np.float32) for a in images]
        rows = (_Texture * max(len(imgs), 1))(*[_Texture(a.shape[1], a.shape[0], a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))) for a in imgs])
        bind = _table(list(bindings), 28)
        keep += [imgs, rows, bind]
        t.textures = ctypes.addressof(rows) if imgs else None; t.n_textures = len(imgs)
        t.material_textures = ctypes.addressof(bind) if len(bindings) else None; t.n_material_textures = len(bindings)
        return cls(_Keep(t, keep), masks=masks)

    def set_textures(self, images, bindings):
        """The arguments of Context.upload_material_textures; clears the masks as the device does."""
        self._imgs = [np.ascontiguousarray(a, np.float32) for a in images]
        self._rows = (_Texture * max(len(self._imgs), 1))(*[_Texture(a.shape[1], a.shape[0], a.ctypes.data_as(ctypes.POINTER(ctypes.c_float)))
                                                            for a in self._imgs])
        self._bind = _table(list(bindings), 28)
        lib().agpt_alpha_oracle_set_textures(self._h, self._rows, c_int(len(self._imgs)), self._bind, c_int(len(bindings)))

    def set_masks(self, masks):
        """The argument of Context.upload_alpha_masks: agpt.alpha_mask(...) rows."""
        masks = list(masks)
        self._masks = _table(masks, 16)
        lib().agpt_alpha_oracle_set_masks(self._h, self._masks if masks else None, c_int(len(masks)))

    def close(self):
        if self._h:
            lib().agpt_alpha_oracle_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def render(self, W, H, first, n, max_depth, depth_arg, threads=0, counters=False):
        out = np.zeros((H, W, 4), np.float32)
        cnt = (ctypes.c_ulonglong * 6)()
        lib().agpt_alpha_oracle_render(self._h, c_int(W), c_int(H), c_int(first), c_int(n), c_int(max_depth), c_int(depth_arg),
                                       c_int(threads or os.cpu_count() or 1), _p(out), cnt)
        return (out, _counters(cnt)) if counters else out

    def li_pixels(self, W, H, xs, ys, ss, max_depth, depth_arg):
        xs, ys, ss = (np.ascontiguousarray(a, np.int32) for a in (xs, ys, ss))
        out = np.zeros((len(xs), 3), np.float32)
        lib().agpt_alpha_oracle_li_pixels(self._h, c_int(W), c_int(H), c_int(len(xs)), _p(xs), _p(ys), _p(ss), c_int(max_depth), c_int(depth_arg), _p(out))
        return out

    def trace_rays(self, rays7, any_hit=False, counters=False):
        """counters: also return the six counters of render (rays_closest, ..., analytic) over these rays."""
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        out = np.zeros(len(rays7), HIT_DTYPE)
        cnt = (ctypes.c_ulonglong * 6)()
        lib().agpt_alpha_oracle_trace_rays(self._h, c_longlong(len(rays7)), _p(rays7), c_int(1 if any_hit else 0), _p(out), cnt)
        return (out, _counters(cnt)) if counters else out

    def primary_hits(self, W, H, sample, counters=False):
        out = np.zeros(W * H, HIT_DTYPE)
        cnt = (ctypes.c_ulonglong * 6)()
        lib().agpt_alpha_oracle_primary_hits(self._h, c_int(W), c_int(H), c_int(sample), _p(out), cnt)
        return (out.reshape(H, W), _counters(cnt)) if counters else out.reshape(H, W)

    def guides(self, W, H, num_samples, threads=0):
        alb = np.zeros((H, W, 4), np.float32)
        nd = np.zeros((H, W, 4), np.float32)
        lib().agpt_alpha_oracle_guides(self._h, c_int(W), c_int(H), c_int(num_samples), c_int(threads or os.cpu_count() or 1), _p(alb), _p(nd))
        return alb, nd
