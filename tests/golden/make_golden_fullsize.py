"""Generate tests/golden/ref_*.npz: what the GPU parity tests (test_gpu_parity, test_gpu_fullsize,
test_gpu_corner_cases) compare against, for checkouts without oracle/_ref.

    python tests/golden/make_golden_fullsize.py

Each file records its `source`: "reference" when oracle/_ref is built (the reference's own integrator,
scene construction included), else "restatement": oracle/agpt_oracle.cpp over the host mirror's scenes,
which tests/test_oracle_port.py and tests/test_host_mirror.py hold bit for bit to the reference's own
fixtures (make_golden.py).  Arrays too large to commit are a fixed, seeded sample of rows (`idx`); the
walk counts are those of the whole table.  The cases are the tests' own; keep the two in step.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import port_binding as port, ref_binding as ref  # noqa: E402
from tests.conftest import load_agpt  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
SAMPLE = 32768
PARITY = [(1, 0, 160, 90), (2, 5, 160, 90), (3, 3, 160, 90), (4, 3, 160, 90), (5, 3, 160, 90), (6, 2, 160, 90), (7, 0, 120, 120)]


class _Restated:
    """RefScene's render / primary_hits / trace_rays answered by the restatement over a host-mirror scene."""

    def __init__(self, agpt, cfg, level):
        self._ps = port.PortScene(agpt.HostScene(cfg, level))

    def render(self, W, H, s0, ns, md, da, crop=None):
        out, cnt = self._ps.render(W, H, s0, ns, md, da, crop=crop)
        return out, cnt["paths"]

    def primary_hits(self, W, H, sample):
        return self._ps.primary_hits(W, H, sample, want_counts=True)

    def trace_rays(self, rays, any_hit=False):
        return self._ps.trace_rays(rays, any_hit)


def sample_rows(n, seed):
    return np.sort(np.random.default_rng(seed).choice(n, min(n, SAMPLE), replace=False))


def crop_box(W, H):
    return (W - 256) // 2, (H - 144) // 2, (W + 256) // 2, (H + 144) // 2


def main():
    agpt = load_agpt()
    source = "reference" if ref.available() else "restatement"
    scene = (lambda c, l: ref.RefScene(c, l)) if ref.available() else (lambda c, l: _Restated(agpt, c, l))

    def save(name, **d):
        np.savez_compressed(os.path.join(OUT, name), source=np.array(source), **d)
        print(name, os.path.getsize(os.path.join(OUT, name)) // 1024, "KB")

    # test_gpu_parity: primary hits of samples 0 and 3, films of 8 spp
    for cfg, level, W, H in PARITY:
        d = agpt.config_defaults(cfg)
        rs = scene(cfg, level)
        h0, _ = rs.primary_hits(W, H, 0)
        h3, _ = rs.primary_hits(W, H, 3)
        acc, _ = rs.render(W, H, 0, 8, d["max_depth"], d["depth_arg"])
        save(f"ref_parity_cfg{cfg}.npz", hits0=h0, hits3=h3, accum=acc[..., :3])
    # test_sphere_run_cull_is_exact: its rays are regenerated from the test's seed
    rs = scene(3, 2)
    rng = np.random.default_rng(20261018)
    n = 120_000
    tgt = np.stack([rng.uniform(-3.7, 3.7, n), rng.uniform(-1.15, 0.15, n), rng.uniform(-4.7, 2.7, n)], 1)
    dist = rng.choice([2.0, 8.0, 40.0, 150.0, 400.0], n)
    dirs = rng.normal(size=(n, 3)); dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    dirs[:, 1] = np.abs(dirs[:, 1]) * rng.choice([1.0, 0.02], n)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    org = tgt + dirs * dist[:, None]
    rays = np.concatenate([org, -dirs, np.full((n, 1), 3.0e38)], 1).astype(np.float32)
    c, _ = rs.trace_rays(rays, any_hit=False)
    a, _ = rs.trace_rays(rays, any_hit=True)
    save("ref_sphere_cull.npz", found=c["found"].astype(np.uint8), prim=c["prim"].astype(np.int16), t=c["t"], found_any=a["found"].astype(np.uint8))
    # test_gpu_fullsize: full-size primary hits (sampled rows, whole-table walk counts)
    for cfg in (2, 3, 5, 4):
        d = agpt.config_defaults(cfg)
        W, H = d["width"], d["height"]
        hits, st = scene(cfg, 0).primary_hits(W, H, 0)
        idx = sample_rows(W * H, cfg)
        save(f"ref_fullsize_hits_cfg{cfg}.npz", idx=idx, hits=hits[idx], walk=np.array([st["interior"], st["boxes"], st["tris"]], np.uint64))
    # centred 256x144 crops of full-size frames
    for cfg, spp in ((3, 4), (4, 2), (5, 4)):
        d = agpt.config_defaults(cfg)
        W, H = d["width"], d["height"]
        x0, y0, x1, y1 = crop_box(W, H)
        want, _ = scene(cfg, 0).render(W, H, 0, spp, d["max_depth"], d["depth_arg"], crop=(x0, y0, x1, y1))
        save(f"ref_crop_cfg{cfg}_{spp}spp.npz", rgb=want[::-1][y0:y1, x0:x1, :3])
    # whole frames (sampled pixels of the film as stored, rows H-1-y)
    frames = [("ref_frame_cfg1_64spp.npz", 1, None, None, 0, 64), ("ref_frame_cfg3_480x270_256spp.npz", 3, 480, 270, 0, 256)]
    frames += [(f"ref_frame_cfg{cfg}_{spp}spp.npz", cfg, None, None, 5, spp) for cfg, spp in ((3, 2), (5, 1), (2, 2))]
    for name, cfg, W, H, s0, spp in frames:
        d = agpt.config_defaults(cfg)
        W, H = W or d["width"], H or d["height"]
        want, _ = scene(cfg, 0).render(W, H, s0, spp, d["max_depth"], d["depth_arg"])
        idx = sample_rows(W * H, cfg * 1000 + spp)
        save(name, idx=idx, rgb=want[..., :3].reshape(-1, 3)[idx])
    # test_cfg8_live_against_reference
    d = agpt.config_defaults(8)
    want, _ = scene(8, 3).render(320, 180, 0, 8, d["max_depth"], d["depth_arg"])
    save("ref_cfg8_live.npz", rgb=want[..., :3])


if __name__ == "__main__":
    main()
