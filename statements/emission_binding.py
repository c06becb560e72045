"""ctypes binding over statements/libagpt_emission_oracle.so -- TEST INFRASTRUCTURE.

EXTENSION: the CPU statement of emissive materials (include/agpt.h agpt_upload_emission), built on the alpha-mask statement
(statements/agpt_emission_oracle.cpp).  EmissionScene takes the tables, alpha masks and emission rows of a host-mirror scene
(HostScene.tables(), HostScene.alpha_masks(), HostScene.emission()); set_textures, set_masks and set_emission replace them as
the device calls do."""
import ctypes
import os
from ctypes import c_int, c_void_p

import numpy as np

from statements import alpha_binding

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libagpt_emission_oracle.so")
_lib = None


def available():
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError(f"{LIB_PATH} missing: run __graft_entry__.build()")
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.agpt_emission_oracle_create.restype = c_void_p
    return _lib


def _p(a):
    return a.ctypes.data_as(c_void_p)


class EmissionScene:
    def __init__(self, host_scene, masks=None, rows=None, rr_by_bounce=False):
        self._keep = host_scene                 # the tables borrow its memory
        masks = host_scene.alpha_masks() if masks is None else list(masks)
        rows = host_scene.emission() if rows is None else list(rows)
        self._masks = alpha_binding._table(masks, 16)
        self._rows = alpha_binding._table(rows, 16)
        self._h = c_void_p(lib().agpt_emission_oracle_create(host_scene.tables(), self._masks if masks else None, c_int(len(masks)),
                                                             self._rows if rows else None, c_int(len(rows))))
        lib().agpt_emission_oracle_set_rr_by_bounce(self._h, c_int(1 if rr_by_bounce else 0))

    def set_textures(self, images, bindings):
        """The arguments of Context.upload_material_textures; clears the masks and the emission rows as the device does."""
        self._imgs = [np.ascontiguousarray(a, np.float32) for a in images]
        self._trows = (alpha_binding._Texture * max(len(self._imgs), 1))(
            *[alpha_binding._Texture(a.shape[1], a.shape[0], a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))) for a in self._imgs])
        self._bind = alpha_binding._table(list(bindings), 28)
        lib().agpt_emission_oracle_set_textures(self._h, self._trows, c_int(len(self._imgs)), self._bind, c_int(len(bindings)))

    def set_masks(self, masks):
        """The argument of Context.upload_alpha_masks: agpt.alpha_mask(...) rows."""
        masks = list(masks)
        self._masks = alpha_binding._table(masks, 16)
        lib().agpt_emission_oracle_set_masks(self._h, self._masks if masks else None, c_int(len(masks)))

    def set_emission(self, rows):
        """The argument of Context.upload_emission: agpt.emission(...) rows."""
        rows = list(rows)
        self._rows = alpha_binding._table(rows, 16)
        lib().agpt_emission_oracle_set_emission(self._h, self._rows if rows else None, c_int(len(rows)))

    def close(self):
        if self._h:
            lib().agpt_emission_oracle_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def render(self, W, H, first, n, max_depth, depth_arg, threads=0, counters=False):
        out = np.zeros((H, W, 4), np.float32)
        cnt = (ctypes.c_ulonglong * 6)()
        lib().agpt_emission_oracle_render(self._h, c_int(W), c_int(H), c_int(first), c_int(n), c_int(max_depth), c_int(depth_arg),
                                          c_int(threads or os.cpu_count() or 1), _p(out), cnt)
        return (out, alpha_binding._counters(cnt)) if counters else out

    def li_pixels(self, W, H, xs, ys, ss, max_depth, depth_arg):
        xs, ys, ss = (np.ascontiguousarray(a, np.int32) for a in (xs, ys, ss))
        out = np.zeros((len(xs), 3), np.float32)
        lib().agpt_emission_oracle_li_pixels(self._h, c_int(W), c_int(H), c_int(len(xs)), _p(xs), _p(ys), _p(ss), c_int(max_depth),
                                             c_int(depth_arg), _p(out))
        return out

    def li_rays(self, rays7, rng_states, max_depth, depth_arg):
        """Context.li_rays with flags 0: rays7 rows (O, D, tmax; D normalised like the Ray ctor), one xorshift32 state per ray."""
        rays7 = np.ascontiguousarray(rays7, np.float32).reshape(-1, 7)
        states = np.ascontiguousarray(rng_states, np.uint32)
        out = np.zeros((len(rays7), 3), np.float32)
        lib().agpt_emission_oracle_li_rays(self._h, c_int(len(rays7)), _p(rays7), _p(states), c_int(max_depth), c_int(depth_arg), _p(out))
        return out
