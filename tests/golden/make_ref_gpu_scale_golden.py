"""Run ON A B200 with oracle/_ref built (oracle/build_ref.sh, from a reference checkout): records the state of the REFERENCE's own
kernels on the benchmark-scale parity scenes of tests/test_gpu_scale.py (scenes.SCALE_CASES), sampled to stay small.

    python tests/golden/make_ref_gpu_scale_golden.py OUTDIR   ->   copy OUTDIR/ref_gpu_<case>.npz into tests/golden/

Per checkpoint: block counts; SHA-256 of the sorted key hashes per block class (scenes.key_digest); maximum and float64 total of
cell mass and momentum over the whole grid; 64 grid blocks (seeded choice, sorted by key); 500 particle states per model (seeded
choice).  The sand column and the fluid dam also record how far the oracle is from the reference over the whole grid: the engine's
tolerance on those scenes is relative to that distance.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import oracle_binding as ob  # noqa: E402
import ref_gpu_binding as rg  # noqa: E402
import scenes  # noqa: E402

GRID_BLOCKS = 64
PARTICLES = 500


def record(sim, nmodels, rng):
    pbc, nbc, ebc = sim.block_counts()
    keys = sim.active_keys()
    out = {"counts": np.array([pbc, nbc, ebc], np.int64)}
    for cls, lo, hi in (("particle", 0, pbc), ("neighbor", pbc, nbc), ("exterior", nbc, ebc)):
        out[f"keys_{cls}"] = np.frombuffer(scenes.key_digest(keys[lo:hi]), np.uint8)
    gh, gg = scenes.grid_by_key(keys, sim.grid())
    out["grid_mass_max"] = np.array([gg[:, 0].max()], np.float64)
    out["grid_mom_absmax"] = np.array([np.abs(gg[:, 1:]).max()], np.float64)
    out["grid_mass_total"] = np.array([gg[:, 0].sum(dtype=np.float64)])
    out["grid_mom_total"] = gg[:, 1:].sum(axis=(0, 2), dtype=np.float64)
    out["grid_mom_abs_total"] = np.array([np.abs(gg[:, 1:]).sum(dtype=np.float64)])
    pick = np.sort(rng.choice(len(gh), size=min(GRID_BLOCKS, len(gh)), replace=False))
    out["grid_sample_keys"], out["grid_sample"] = gh[pick], gg[pick]
    for m in range(nmodels):
        st = sim.particle_state(m)
        out[f"state{m}_count"] = np.array([len(st)], np.int64)
        out[f"state{m}_sample"] = st[np.sort(rng.choice(len(st), size=min(PARTICLES, len(st)), replace=False))]
    return out


def grid_deviation(a, b):
    """(max |cell mass a - b| / max mass, max |cell momentum a - b| / max |momentum|) of two simulators aligned by block key."""
    ha, ga = scenes.grid_by_key(a.active_keys(), a.grid())
    hb, gb = scenes.grid_by_key(b.active_keys(), b.grid())
    assert np.array_equal(ha, hb)
    return float(np.abs(ga[:, 0] - gb[:, 0]).max() / ga[:, 0].max()), float(np.abs(ga[:, 1:] - gb[:, 1:]).max() / np.abs(ga[:, 1:]).max())


def main(outdir):
    os.makedirs(outdir, exist_ok=True)
    for name, (make, checkpoints) in scenes.SCALE_CASES.items():
        scene = make()
        ref = rg.build_ref(scene)
        osim = None
        if name != "spheres5m":
            osim = scenes.build_oracle(ob, scene, max_blocks=scenes.max_blocks_for(scene, 4.0), threads=min(os.cpu_count() or 1, 32))
        rng = np.random.default_rng(1)
        data, done = {}, 0
        for cp in checkpoints:
            ref.step(cp - done)
            if osim is not None:
                osim.step(cp - done)
                data[f"s{cp}_ref_oracle_deviation"] = np.array(grid_deviation(ref, osim))
            done = cp
            for k, v in record(ref, len(scene["models"]), rng).items():
                data[f"s{cp}_{k}"] = v
        ref.close()
        if osim is not None:
            osim.close()
        np.savez_compressed(os.path.join(outdir, f"ref_gpu_{name}.npz"), **data)
        print(name, {k: v.shape for k, v in data.items()}, flush=True)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
