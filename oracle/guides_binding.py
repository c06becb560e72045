"""ctypes binding over oracle/libagpt_guides_oracle.so -- TEST INFRASTRUCTURE.

EXTENSION: the CPU statement of the denoiser's guide buffers (include/agpt.h agpt_render_guides), built on the oracle
(oracle/agpt_guides_oracle.cpp).  GuideScene takes the same tables as port_binding.PortScene."""
import ctypes
import os
from ctypes import c_int, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libagpt_guides_oracle.so")
# agpt_guide_sample
SAMPLE_DTYPE = np.dtype([("albedo", np.float32, 3), ("normal", np.float32, 3), ("dir", np.float32, 3), ("t", np.float32), ("prim", np.int32)])
_lib = None


def available():
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError(f"{LIB_PATH} missing: run __graft_entry__.build()")
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.agpt_oracle_scene_create.restype = c_void_p
    return _lib


class GuideScene:
    """The statement fed with the flattened tables of a host-mirror scene (HostScene.tables())."""

    def __init__(self, host_scene):
        self._keep = host_scene                 # the tables borrow its memory
        self._h = c_void_p(lib().agpt_oracle_scene_create(host_scene.tables()))

    def close(self):
        if self._h:
            lib().agpt_oracle_scene_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def guides(self, W, H, num_samples, threads=0):
        """(per-sample records [num_samples, H*W] with image row y at y*W + x, albedo [H, W, 4], normal_depth [H, W, 4]), the
        last two in the film's row order as agpt_read_guides returns them."""
        per = np.zeros((num_samples, W * H), SAMPLE_DTYPE)
        alb = np.zeros((H, W, 4), np.float32)
        nd = np.zeros((H, W, 4), np.float32)
        fp = lambda a: a.ctypes.data_as(c_void_p)
        lib().agpt_guides_oracle(self._h, c_int(W), c_int(H), c_int(num_samples), c_int(threads or os.cpu_count() or 1), fp(per), fp(alb), fp(nd))
        return per, alb, nd
