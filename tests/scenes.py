"""Test-side scene helpers: everything of claymore_b200.scenes plus the oracle builders (tests only)."""
import hashlib

import numpy as np

from claymore_b200.scenes import *  # noqa: F401,F403
from claymore_b200.scenes import material_parameters
from claymore_b200 import scenes as _pkg

J_FLUID, FIXED_COROTATED, SAND, NACC = 0, 1, 2, 3


def apply_material(sim, model_id, material, dx, is_oracle):
    """Engine: keyword `model`; oracle binding: model id first."""
    name, args = material_parameters(material, dx)
    if is_oracle:
        getattr(sim, name)(model_id, *args)
    else:
        getattr(sim, name)(*args, model=model_id)


def build_oracle(ob, scene, dt=1e-4, max_blocks=4000, max_ppc=128, threads=1, cfl=0.5):
    cfg = ob.make_config(domain_bits=scene["domain_bits"], max_ppc=max_ppc, cfl=cfl)
    sim = ob.OracleSim(cfg, dt, max_blocks, threads=threads)
    dx = 1.0 / (1 << scene["domain_bits"])
    for m in scene["models"]:
        mid = sim.init_model(m["material"], m["pos"], m["v0"])
        apply_material(sim, mid, m["material"], dx, True)
    sim.initial_setup()
    return sim


def match_particles(a, b, tol):
    """Bijective nearest-neighbour match of two particle sets by position; returns index array into b."""
    from scipy.spatial import cKDTree
    d, idx = cKDTree(b[:, :3]).query(a[:, :3], k=1)
    assert d.max() <= tol, f"unmatched particle: nearest distance {d.max():.3e} > {tol:.3e}"
    assert len(np.unique(idx)) == len(a), "particle match is not a bijection"
    return idx


def key_digest(keys):
    """SHA-256 of a block key set (order-free): compares key sets of tens of thousands of blocks against a 32-byte record."""
    return hashlib.sha256(np.sort(key_hash(keys)).astype("<i8").tobytes()).digest()


# benchmark-scale parity scenes of tests/test_gpu_scale.py: name -> (scene builder, checkpoints in sub-steps)
SCALE_CASES = {
    "spheres5m": (lambda: workload("spheres5m")[0], (1, 20, 100)),
    "sand2m_512": (lambda: sand_column(domain_bits=9, size=(50, 100, 50)), (1, 20)),
    "fluid1m_512": (lambda: fluid_dam(domain_bits=9, size=(64, 40, 64), base=(12, 12, 12)), (1, 20)),
}
