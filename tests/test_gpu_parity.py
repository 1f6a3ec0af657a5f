"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on identical seeded inputs.

Tolerances (FP32, stated per SURVEY.md section 8c): active-block key sets and block counts bit-exact; per-cell grid mass
rel 1e-5 (+ abs floor), momentum abs 1e-4 * max|mv|; particle positions 1e-6 absolute (domain is [0,1]^3), F 2e-5.
"""
import ctypes as C

import numpy as np
import pytest

import scenes

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _compare_state(osim, esim, nmodels, steps_label, pos_tol=2e-6, f_tol=5e-5):
    # block counts and key sets: bit-exact
    st = esim.stats()
    assert st.error == 0, f"engine error bits {st.error} {steps_label}"
    opb, onb, oeb = osim.block_counts()
    assert (st.particle_block_count, st.neighbor_block_count, st.exterior_block_count) == (opb, onb, oeb), steps_label
    okeys, ekeys = osim.active_keys(), esim.active_keys()
    for lo, hi in ((0, opb), (opb, onb), (onb, oeb)):  # per class: particle / neighbour / exterior
        assert np.array_equal(np.sort(scenes.key_hash(okeys[lo:hi])), np.sort(scenes.key_hash(ekeys[lo:hi]))), f"key set mismatch in class [{lo},{hi}) {steps_label}"
    # grid: per cell, aligned by key
    oh, og = scenes.grid_by_key(okeys, osim.grid())
    eh, eg = scenes.grid_by_key(ekeys, esim.grid())
    assert np.array_equal(oh, eh)
    mass_o, mass_e = og[:, 0], eg[:, 0]
    assert np.allclose(mass_e, mass_o, rtol=1e-5, atol=1e-5 * mass_o.max()), f"grid mass {steps_label}: {np.abs(mass_e - mass_o).max():.3e}"
    mom_scale = np.abs(og[:, 1:]).max()
    assert np.abs(eg[:, 1:] - og[:, 1:]).max() <= 1e-4 * mom_scale, f"grid momentum {steps_label}: {np.abs(eg[:, 1:] - og[:, 1:]).max():.3e} vs scale {mom_scale:.3e}"
    assert abs(mass_e.sum(dtype=np.float64) - mass_o.sum(dtype=np.float64)) <= 1e-6 * mass_o.sum(dtype=np.float64)
    # particles: matched by position
    for m in range(nmodels):
        so, se = osim.particle_state(m), esim.particle_state(m)
        assert len(so) == len(se), f"particle count model {m} {steps_label}"
        idx = scenes.match_particles(so, se, tol=pos_tol)
        se = se[idx]
        assert np.abs(se[:, :3] - so[:, :3]).max() <= pos_tol
        if so.shape[1] > 3:
            assert np.abs(se[:, 3:] - so[:, 3:]).max() <= f_tol, f"particle state model {m} {steps_label}: {np.abs(se[:, 3:] - so[:, 3:]).max():.3e}"


@pytest.mark.parametrize("material", [scenes.FIXED_COROTATED, scenes.J_FLUID, scenes.SAND, scenes.NACC])
@pytest.mark.parametrize("use_graph", [False, True])
def test_engine_matches_oracle_small_cube(oracle, cuda_lib, material, use_graph):
    if use_graph and material not in (scenes.FIXED_COROTATED,):
        pytest.skip("graph replay is material independent; covered once")
    scene = scenes.small_cube(material=material)
    osim = scenes.build_oracle(oracle, scene)
    esim = scenes.build_engine(scene, use_graph=use_graph)
    _compare_state(osim, esim, 1, "after setup")
    for k in range(3):
        osim.step(5)
        esim.step(5)
        _compare_state(osim, esim, 1, f"after {5 * (k + 1)} steps")
    assert abs(esim.stats().dt - osim.dt) <= 1e-9
    esim.close()


def test_engine_two_models_colliding(oracle, cuda_lib):
    scene = scenes.two_cubes_colliding()
    osim = scenes.build_oracle(oracle, scene, dt=2e-4)
    esim = scenes.build_engine(scene, dt=2e-4)
    for k in range(4):
        osim.step(10)
        esim.step(10)
        _compare_state(osim, esim, 2, f"after {10 * (k + 1)} steps", pos_tol=5e-6, f_tol=2e-4)
    esim.close()


def test_engine_jittered_positions(oracle, cuda_lib):
    scene = scenes.small_cube(jitter_seed=3)
    osim = scenes.build_oracle(oracle, scene)
    esim = scenes.build_engine(scene)
    osim.step(8)
    esim.step(8)
    _compare_state(osim, esim, 1, "jittered, 8 steps")
    esim.close()


def test_engine_small_max_ppc(oracle, cuda_lib):
    """max_ppc is a runtime parameter here (compile-time 128 in the reference): tags / strides must follow it."""
    scene = scenes.small_cube()
    osim = scenes.build_oracle(oracle, scene, max_ppc=32)
    esim = scenes.build_engine(scene, max_ppc=32)
    osim.step(6)
    esim.step(6)
    _compare_state(osim, esim, 1, "max_ppc=32, 6 steps")
    esim.close()


def test_jelly_cube_config1(oracle, cuda_lib):
    """BASELINE config 1: 128^3 grid, 140 608-particle jelly cube, fixed-corotated."""
    scene = scenes.jelly_cube()
    osim = scenes.build_oracle(oracle, scene, threads=8)
    esim = scenes.build_engine(scene)
    n = sum(len(m["pos"]) for m in scene["models"])
    assert n == 140608
    osim.step(10)
    esim.step(10)
    _compare_state(osim, esim, 1, "config1, 10 steps")
    # invariants at full size: particle count and mass conservation
    assert len(esim.retrieve(0)) == n
    g = esim.grid()
    dx = 1.0 / 128
    assert abs(g[:, 0].sum(dtype=np.float64) - n * 1e3 * dx ** 3 / 8) <= 1e-5 * n * 1e3 * dx ** 3 / 8
    esim.close()


# ---- kernel-level differential test through the drop-in entry points --------------------------------------
def _dev(torch, arr):
    return torch.from_numpy(np.ascontiguousarray(arr)).cuda()


def _cb_buffer(cb, ob_struct, t):
    pb = cb.ParticleBuffer()
    for f, _ in cb.ParticleBuffer._fields_:
        if f in t:
            setattr(pb, f, t[f].data_ptr())
        elif hasattr(ob_struct, f):
            setattr(pb, f, getattr(ob_struct, f))
    return pb


@pytest.mark.parametrize("material", [scenes.FIXED_COROTATED, scenes.J_FLUID, scenes.SAND])
def test_g2p2g_kernel_differential(oracle, cuda_lib, material):
    """Same containers in, same containers out: cb200_g2p2g vs orc_g2p2g after a few warm-up steps (deformed F)."""
    torch = _torch()
    import claymore_b200 as cb
    ob = oracle
    scene = scenes.small_cube(material=material)
    osim = scenes.build_oracle(ob, scene)
    osim.step(4)
    pbc, nbc, ebc = osim.block_counts()
    cfg_o = osim.cfg
    cfg_c = cb.Config(domain_bits=cfg_o.domain_bits, max_ppc=cfg_o.max_ppc)
    dt = osim.dt
    # grid[0] currently holds mass/momentum: turn it into velocities exactly as the step would
    cur, nxt = osim.buffer_arrays(0, 0), osim.buffer_arrays(0, 1)
    part, prev = osim.partition_arrays(0), osim.partition_arrays(1)
    g0, g1 = osim.grid_array(0), osim.grid_array(1)
    mv = np.zeros(1, np.float32)
    ob.lib().orc_update_grid_velocity_query_max(C.byref(cfg_o), nbc, ob.ptr(g0), part["struct"], dt, ob.ptr(mv))
    g1[: nbc * 256] = 0
    nxt["cell_particle_counts"][: ebc * 64] = 0
    keys = ("bins", "cell_particle_counts", "particle_bucket_sizes", "cellbuckets", "blockbuckets", "bin_offsets")
    t_cur = {k: _dev(torch, cur[k]) for k in keys}
    t_nxt = {k: _dev(torch, nxt[k]) for k in keys}
    t_part = {k: _dev(torch, part[k]) for k in ("count", "index_table", "active_keys")}
    t_prev = {k: _dev(torch, prev[k]) for k in ("count", "index_table", "active_keys")}
    t_g0, t_g1 = _dev(torch, g0), _dev(torch, g1)
    c_cur, c_nxt = _cb_buffer(cb, cur["struct"], t_cur), _cb_buffer(cb, nxt["struct"], t_nxt)
    c_part, c_prev = cb.Partition(), cb.Partition()
    for name, t in (("count", "count"), ("index_table", "index_table"), ("active_keys", "active_keys")):
        setattr(c_part, name, t_part[t].data_ptr())
        setattr(c_prev, name, t_prev[t].data_ptr())
    new_dt = dt
    err = cuda_lib.cb200_g2p2g(C.byref(cfg_c), dt, new_dt, pbc, c_cur, c_nxt, c_prev, c_part, t_g0.data_ptr(), t_g1.data_ptr(), None)
    assert err == 0
    torch.cuda.synchronize()
    ob.lib().orc_g2p2g(C.byref(cfg_o), dt, new_dt, pbc, cur["struct"], nxt["struct"], prev["struct"], part["struct"], ob.ptr(g0), ob.ptr(g1))
    # next bins: slot-for-slot (same bucket order in, same slots out)
    bins_c, bins_o = t_nxt["bins"].cpu().numpy(), nxt["bins"]
    bf = ob.BIN_FLOATS[material]
    nch = ob.CHANNELS[material]
    offs, sizes = nxt["bin_offsets"], nxt["particle_bucket_sizes"]
    worst_pos = worst_f = 0.0
    for b in range(pbc):
        n = int(sizes[b])
        for bi in range((n + 31) // 32):
            lanes = min(32, n - 32 * bi)
            o = (int(offs[b]) + bi) * bf
            a = bins_c[o:o + nch * 32].reshape(nch, 32)[:, :lanes]
            r = bins_o[o:o + nch * 32].reshape(nch, 32)[:, :lanes]
            worst_pos = max(worst_pos, np.abs(a[:3] - r[:3]).max())
            if nch > 3:
                worst_f = max(worst_f, np.abs(a[3:] - r[3:]).max())
    assert worst_pos <= 1e-6, worst_pos
    assert worst_f <= 2e-5, worst_f
    # re-bucketing: cell counts exact, tags equal as sets per cell
    cc_c, cc_o = t_nxt["cell_particle_counts"].cpu().numpy()[: ebc * 64], nxt["cell_particle_counts"][: ebc * 64]
    assert np.array_equal(cc_c, cc_o)
    cb_c, cb_o = t_nxt["cellbuckets"].cpu().numpy(), nxt["cellbuckets"]
    mp = cfg_o.max_ppc
    for cell in np.nonzero(cc_o)[0]:
        n = cc_o[cell]
        assert np.array_equal(np.sort(cb_c[cell * mp: cell * mp + n]), np.sort(cb_o[cell * mp: cell * mp + n]))
    # next grid per cell
    gc, go = t_g1.cpu().numpy()[: nbc * 256].reshape(nbc, 4, 64), g1[: nbc * 256].reshape(nbc, 4, 64)
    assert np.allclose(gc[:, 0], go[:, 0], rtol=1e-5, atol=1e-5 * go[:, 0].max())
    assert np.abs(gc[:, 1:] - go[:, 1:]).max() <= 1e-4 * np.abs(go[:, 1:]).max()


def test_grid_update_kernel_differential(oracle, cuda_lib):
    torch = _torch()
    import claymore_b200 as cb
    ob = oracle
    scene = scenes.small_cube()
    osim = scenes.build_oracle(ob, scene)
    osim.step(3)
    _, nbc, _ = osim.block_counts()
    cfg_o = osim.cfg
    cfg_c = cb.Config(domain_bits=cfg_o.domain_bits, max_ppc=cfg_o.max_ppc)
    part = osim.partition_arrays(0)
    g0 = osim.grid_array(0)
    t_g = _dev(torch, g0)
    t_keys = _dev(torch, part["active_keys"])
    t_mv = torch.zeros(1, device="cuda")
    c_part = cb.Partition()
    c_part.active_keys = t_keys.data_ptr()
    assert cuda_lib.cb200_update_grid_velocity_query_max(C.byref(cfg_c), nbc, t_g.data_ptr(), c_part, osim.dt, t_mv.data_ptr(), None) == 0
    torch.cuda.synchronize()
    mv = np.zeros(1, np.float32)
    ob.lib().orc_update_grid_velocity_query_max(C.byref(cfg_o), nbc, ob.ptr(g0), part["struct"], osim.dt, ob.ptr(mv))
    gc = t_g.cpu().numpy()[: nbc * 256]
    assert np.allclose(gc, g0[: nbc * 256], rtol=1e-6, atol=1e-7)
    assert abs(float(t_mv.item()) - float(mv[0])) <= 1e-6 * max(1.0, float(mv[0]))


# ---- MGSP: two particle shards, exchange through peer inboxes (both ranks on ONE GPU, one host thread each) -----------
@pytest.mark.timeout(300)
@pytest.mark.parametrize("v0,dt_default", [((0.3, -1.0, 0.2), 1e-4), ((1.0, -10.0, 0.5), 1e-3)], ids=["dt_default_binds", "cfl_binds"])
def test_mgsp_two_shards_match_single_domain(oracle, cuda_lib, v0, dt_default):
    """cfl_binds: dt follows the max grid velocity, so the ranks must agree on the all-reduced maximum bit for bit."""
    import threading
    from claymore_b200 import mgsp
    scene = scenes.small_cube(v0=v0)
    osim = scenes.build_oracle(oracle, scene, dt=dt_default)
    sims = []
    for r in range(2):
        part = mgsp.partition_scene(scene, r, 2)
        sims.append(mgsp.build_rank_sim(part, r, 2, dt_default, 4000, scenes.apply_material))
    ptrs = [s.mgsp_inbox() for s in sims]
    for s in sims:
        s.mgsp_set_peers(ptrs)
    # initial_setup synchronises with the peer (halo tagging), so the two ranks need a host thread each, as in the
    # reference (one worker thread per GPU, mgsp_benchmark.cuh:309-334)
    errs = []

    def run(s):
        try:
            s.initial_setup()
        except Exception as e:  # pragma: no cover
            errs.append(e)
    th = [threading.Thread(target=run, args=(s,)) for s in sims]
    [t.start() for t in th]
    [t.join(120) for t in th]
    assert not errs and not any(t.is_alive() for t in th)

    def check(label):
        okeys, ogrid = osim.active_keys(), osim.grid()
        oh, og = scenes.grid_by_key(okeys, ogrid)
        lut = {int(h): i for i, h in enumerate(oh)}
        total = np.zeros_like(og)
        seen = np.zeros(len(og), bool)
        shared_sets = []
        for s in sims:
            st = s.stats()
            assert st.error == 0, (label, st.error)
            k, g = s.active_keys(), s.grid()
            shared_sets.append(set(int(h) for h in scenes.key_hash(k[: len(g)])))
        common = shared_sets[0] & shared_sets[1]
        assert len(common) > 0
        scale = np.abs(og).max(axis=(0, 2), keepdims=True)
        for s in sims:
            k, g = s.active_keys(), s.grid()
            for b, h in enumerate(scenes.key_hash(k[: len(g)])):
                i = lut.get(int(h))
                if i is None:
                    assert np.abs(g[b]).max() == 0, label
                    continue
                if int(h) in common:   # halo block: both owners hold the full sum
                    assert np.all(np.abs(g[b] - og[i]) <= 2e-4 * scale[0] + 1e-12), (label, "halo block differs from the single-domain block")
                    if not seen[i]:
                        total[i] = g[b]
                else:
                    total[i] += g[b]
                seen[i] = True
        assert np.all(np.abs(total - og) <= 2e-4 * scale + 1e-12), label
        # particles: union of the shards == single domain
        so = osim.particle_state(0)
        se = np.concatenate([s.particle_state(0) for s in sims])
        assert len(so) == len(se)
        loose = dt_default > 5e-4   # 8x larger sub-steps in the CFL-bound variant
        idx = scenes.match_particles(so, se, tol=2e-5 if loose else 3e-6)
        assert np.abs(se[idx][:, 3:] - so[:, 3:]).max() <= (1e-3 if loose else 1e-4), (label, np.abs(se[idx][:, 3:] - so[:, 3:]).max())
        assert abs(sims[0].stats().dt - sims[1].stats().dt) == 0.0
        # when the CFL bound binds, dt inherits the ~1e-6 relative summation-order noise of the grid velocities
        assert abs(sims[0].stats().dt - osim.dt) <= 1e-4 * osim.dt, (sims[0].stats().dt, osim.dt)
        if dt_default > 5e-4:
            assert osim.dt < dt_default  # the CFL bound is the one that binds in this variant

    check("after setup")
    for k in range(3):
        osim.step(4)
        for s in sims:
            s.step(4)
        for s in sims:
            s.sync()
        check(f"after {4 * (k + 1)} steps")
    shared, halo_pb = sims[0].mgsp_halo_counts()
    assert shared[1] > 0 and halo_pb > 0
    for s in sims:
        s.close()


# ---- the CUDA path against outputs of the reference's OWN kernels (fixtures recorded on a B200, tests/golden/) ----------
@pytest.mark.parametrize("name", ["fc_small_cube", "fluid_small_cube", "sand_small_cube", "fc_two_cubes"])
def test_engine_matches_reference_gpu_golden(cuda_lib, name):
    import os
    from test_oracle_cpu import REF_GPU_CASES, compare_with_ref_gpu_golden
    make, dt = REF_GPU_CASES[name]
    scene = make()
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"ref_gpu_{name}.npz"))
    sim = scenes.build_engine(scene, dt=dt)
    done = 0
    for cp in (0, 1, 5, 15):
        sim.step(cp - done)
        done = cp
        assert sim.stats().error == 0
        compare_with_ref_gpu_golden(sim, g, cp, len(scene["models"]), f"{name} step {cp}")
    sim.close()


def test_reference_gpu_live_three_way(oracle, cuda_lib):
    """Reference (its state recorded on a B200, tests/golden/ref_gpu_fc_jitter_cube.npz), oracle and engine side by side on a
    jittered scene that the other fixtures do not cover."""
    import os
    from test_oracle_cpu import compare_with_ref_gpu_golden
    scene = scenes.small_cube(jitter_seed=11)
    golden = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_gpu_fc_jitter_cube.npz"))
    osim = scenes.build_oracle(oracle, scene)
    esim = scenes.build_engine(scene)
    for s in (osim, esim):
        s.step(10)
    compare_with_ref_gpu_golden(osim, golden, 10, 1, "oracle vs reference")
    compare_with_ref_gpu_golden(esim, golden, 10, 1, "engine vs reference")
    esim.close()


def test_advance_frame_matches_reference_frame_loop(oracle, cuda_lib):
    """main_loop's inner for-loop (gmpm_simulator.cuh:324): sub-steps until the frame time is reached, the last dt clamped."""
    scene = scenes.small_cube()
    fps, dt = 240, 1e-4
    frame = np.float32(1.0 / fps)
    osim = scenes.build_oracle(oracle, scene, dt=dt)
    esim = scenes.build_engine(scene, dt=dt, fps=fps)
    for f in range(2):
        t, steps = np.float32(0.0), 0
        while t < frame:
            osim.step(1, time_left=float(frame - t))
            t = np.float32(t + np.float32(osim.dt))
            steps += 1
        taken = esim.advance_frame()
        assert taken == steps == 42, (taken, steps)
        st = esim.stats()
        assert st.error == 0 and abs(st.dt - osim.dt) <= 1e-9 and abs(st.step_time - float(frame)) <= 1e-7
        _compare_state(osim, esim, 1, f"after frame {f + 1}", pos_tol=5e-6, f_tol=2e-4)
    esim.close()


def test_engine_dense_blocks_multiple_passes(oracle, cuda_lib):
    """27 particles per cell = 1728 per particle block: g2p2g stages such a block in four 512-particle passes that share one
    accumulation arena (reference: one CUDA block strides over the whole bucket, `particle_id_in_block += blockDim.x`, mgmpm_kernels.cuh:746)."""
    scene = scenes.dense_cube()
    osim = scenes.build_oracle(oracle, scene)
    esim = scenes.build_engine(scene)
    _compare_state(osim, esim, 1, "dense, after setup")
    for k in range(2):
        osim.step(4)
        esim.step(4)
        _compare_state(osim, esim, 1, f"dense, after {4 * (k + 1)} steps", pos_tol=5e-6, f_tol=2e-4)
    esim.close()
