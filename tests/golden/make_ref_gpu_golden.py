"""Run ON A B200: records outputs of the REFERENCE's own kernels (oracle/_ref/libclaymore_ref_gpu_d6.so, built from a reference
checkout by oracle/build_ref.sh) on the seeded test scenes, in an order-free form, as golden fixtures.

    python tests/golden/make_ref_gpu_golden.py OUTDIR [CASE ...]   ->   copy OUTDIR/ref_gpu_<case>.npz into tests/golden/

Fixture content per scene and checkpoint: block counts; sorted key hashes per block class; grid blocks (mass + momentum)
sorted by key; particle states sorted lexicographically by quantised position (ties cannot occur: lattice spacing dx/2).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import ref_gpu_binding as rg  # noqa: E402
import scenes  # noqa: E402

CHECKPOINTS = (0, 1, 5, 15)
# name -> (scene, dt, checkpoints)
CASES = {
    "fc_small_cube": (lambda: scenes.small_cube(material=scenes.FIXED_COROTATED), 1e-4, CHECKPOINTS),
    "fluid_small_cube": (lambda: scenes.small_cube(material=scenes.J_FLUID), 1e-4, CHECKPOINTS),
    "sand_small_cube": (lambda: scenes.small_cube(material=scenes.SAND), 1e-4, CHECKPOINTS),
    "fc_two_cubes": (scenes.two_cubes_colliding, 2e-4, CHECKPOINTS),
    "fc_jitter_cube": (lambda: scenes.small_cube(jitter_seed=11), 1e-4, (10,)),   # test_gpu_parity.py three-way test
}


def snapshot(sim, nmodels):
    pbc, nbc, ebc = sim.block_counts()
    keys = sim.active_keys()
    h = scenes.key_hash(keys)
    out = {"counts": np.array([pbc, nbc, ebc]), "keys_particle": np.sort(h[:pbc]), "keys_neighbor": np.sort(h[pbc:nbc]), "keys_exterior": np.sort(h[nbc:ebc])}
    gh, gg = scenes.grid_by_key(keys, sim.grid())
    out["grid_keys"], out["grid"] = gh, gg
    for m in range(nmodels):
        st = sim.particle_state(m)
        q = np.round(st[:, :3] * 1e5).astype(np.int64)
        out[f"state{m}"] = st[np.lexsort((q[:, 2], q[:, 1], q[:, 0]))]
    out["dt"] = np.array([sim.dt], np.float32)
    return out


def main(outdir, names):
    os.makedirs(outdir, exist_ok=True)
    for name in names:
        make, dt, checkpoints = CASES[name]
        scene = make()
        sim = rg.build_ref(scene, dt)
        data, done = {}, 0
        for cp in checkpoints:
            sim.step(cp - done)
            done = cp
            for k, v in snapshot(sim, len(scene["models"])).items():
                data[f"s{cp}_{k}"] = v
        sim.close()
        np.savez_compressed(os.path.join(outdir, f"ref_gpu_{name}.npz"), **data)
        print(name, {k: v.shape for k, v in data.items() if k.startswith(f"s{checkpoints[-1]}_")})


if __name__ == "__main__":
    if len(sys.argv) < 2:
        raise SystemExit(__doc__)
    main(sys.argv[1], sys.argv[2:] or sorted(CASES))
