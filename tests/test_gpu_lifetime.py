"""GPU: what a refused call leaves resident (include/agpt.h: a refused upload leaves the old scene intact)."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


class Envmap(ctypes.Structure):  # agpt_envmap
    _fields_ = [("width", ctypes.c_int32), ("height", ctypes.c_int32), ("rgb", ctypes.c_void_p), ("func", ctypes.c_void_p),
                ("cdf", ctypes.c_void_p), ("func_int", ctypes.c_float)]


def test_refused_envmap_keeps_the_resident_one(agpt, gpu_ctx):
    """cfg 7 is lit by an InfiniteAreaLight.  A malformed map (width -1) is refused with AGPT_ERR_INVALID, and the scene still
    renders with the map it had: the same film, bit for bit."""
    W, H, spp = 64, 36, 2
    d = agpt.config_defaults(7)
    hs = agpt.HostScene(7, 0)
    hs.upload(gpu_ctx)
    gpu_ctx.set_film(W, H)

    def render():
        gpu_ctx.clear()
        gpu_ctx.render(0, spp, d["max_depth"], d["depth_arg"])
        return gpu_ctx.read_accum().copy()

    film = render()
    assert film[..., :3].max() > 0
    bad = Envmap(-1, 1, None, None, None, 0.0)
    assert agpt.core().agpt_upload_envmap(gpu_ctx.handle, ctypes.byref(bad)) == -1      # AGPT_ERR_INVALID
    assert np.array_equal(render().view(np.uint32), film.view(np.uint32))
