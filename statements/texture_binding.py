"""ctypes binding over statements/libagpt_texture_oracle.so -- TEST INFRASTRUCTURE.

EXTENSION: the CPU statement of image textures on the base colour of Disney materials (include/agpt.h
agpt_upload_textures), built on the oracle (statements/agpt_texture_oracle.cpp).  TextureScene takes the tables of a
host-mirror scene (HostScene.tables()), texture bindings included."""
import ctypes
import os
from ctypes import c_int, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libagpt_texture_oracle.so")
_lib = None


def available():
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError(f"{LIB_PATH} missing: run __graft_entry__.build()")
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.agpt_texture_oracle_create.restype = c_void_p
    return _lib


def _p(a):
    return a.ctypes.data_as(c_void_p)


def lookup(image, uv):
    """The statement's bilinear lookup: image (H, W, 3) float32, uv (n, 2) float32 -> (n, 3) float32."""
    image = np.ascontiguousarray(image, np.float32)
    uv = np.ascontiguousarray(uv, np.float32).reshape(-1, 2)
    out = np.zeros((len(uv), 3), np.float32)
    lib().agpt_texture_oracle_lookup(c_int(image.shape[1]), c_int(image.shape[0]), _p(image), c_int(len(uv)), _p(uv), _p(out))
    return out


def atan2f(y, x):
    """fdlibm e_atan2f.c in float, as the device states the sphere's u with."""
    y = np.ascontiguousarray(y, np.float32).ravel()
    x = np.ascontiguousarray(x, np.float32).ravel()
    out = np.zeros(len(y), np.float32)
    lib().agpt_texture_oracle_atan2(c_int(len(y)), _p(y), _p(x), _p(out))
    return out


class TextureScene:
    def __init__(self, host_scene, rr_by_bounce=False):
        self._keep = host_scene                 # the tables borrow its memory
        self._h = c_void_p(lib().agpt_texture_oracle_create(host_scene.tables()))
        lib().agpt_texture_oracle_set_rr_by_bounce(self._h, c_int(1 if rr_by_bounce else 0))

    def close(self):
        if self._h:
            lib().agpt_texture_oracle_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def render(self, W, H, first, n, max_depth, depth_arg, threads=0):
        """H x W float4 film (film row order) of samples [first, first + n), as agpt_render adds them."""
        out = np.zeros((H, W, 4), np.float32)
        lib().agpt_texture_oracle_render(self._h, c_int(W), c_int(H), c_int(first), c_int(n), c_int(max_depth), c_int(depth_arg),
                                         c_int(threads or os.cpu_count() or 1), _p(out))
        return out

    def li_pixels(self, W, H, xs, ys, ss, max_depth, depth_arg):
        xs, ys, ss = (np.ascontiguousarray(a, np.int32) for a in (xs, ys, ss))
        out = np.zeros((len(xs), 3), np.float32)
        lib().agpt_texture_oracle_li_pixels(self._h, c_int(W), c_int(H), c_int(len(xs)), _p(xs), _p(ys), _p(ss), c_int(max_depth), c_int(depth_arg), _p(out))
        return out

    def guides(self, W, H, num_samples, threads=0):
        alb = np.zeros((H, W, 4), np.float32)
        nd = np.zeros((H, W, 4), np.float32)
        lib().agpt_texture_oracle_guides(self._h, c_int(W), c_int(H), c_int(num_samples), c_int(threads or os.cpu_count() or 1), _p(alb), _p(nd))
        return alb, nd

    def hit_uv(self, rays7):
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        out = np.zeros((len(rays7), 3), np.float32)
        lib().agpt_texture_oracle_hit_uv(self._h, c_int(len(rays7)), _p(rays7), _p(out))
        return out
