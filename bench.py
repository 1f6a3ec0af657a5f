#!/usr/bin/env python
"""bench.py -- particle-steps/s of the fused G2P2G + sparse-grid partition/update sub-step (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W                  (N>1: launched under torch.distributed.run)
  python bench.py --impl reference ...                           CPU arm: the oracle port on the host cores

Workload (--workload, default spheres40m): the scene BASELINE.json's north_star quotes its target on -- GMPM two elastic
spheres (fixed-corotated), 512^3 grid, 40 M particles.  N=1 runs it on one B200 and adds, in the same process,
  * `ref_gpu`: the REFERENCE's own kernels (oracle/_ref/libclaymore_ref_gpu_d<bits>.so, built unmodified for sm_100a) on the same
    scene on the same GPU -- the denominator of the ">= 2x reference claymore per GPU" target,
  * `configs1`: the device-timed value of BASELINE configs[1] (5 M particles, 256^3),
  * `cpu_baseline`: the oracle port (OpenMP) on the host cores on a bounded sample.
N>1: MGSP static particle partition of the SAME scene (strong scaling): the particles are cut into N equal-count x-slabs, one
process per GPU; halo grid blocks are reduced by g2p2g itself over NVLink (CUDA-IPC peer memory).  The line carries `parity`:
the union of the shards compared with a single-GPU run of the same scene on rank 0 (block key sets, per-cell mass / momentum,
totals) and the agreement of the owners of every shared grid block.  --scaling weak keeps the round-1 weak-scaling run (5 M per rank).
A "step" is one sub-step (grid update, g2p2g, partition rebuild) with fixed dt (default_dt 1e-4; the CFL bound never binds).
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "million particle-steps/sec"
UNIT = "Mparticle-steps/s"
BLOCK_BYTES_G2P2G = 2048.0      # per particle block: 768 B velocity read + 1024 B accumulate-write + 256 B cell counters (SURVEY.md 8d)
BYTES_BY_MATERIAL = {0: 40.0, 1: 104.0, 2: 112.0, 3: 112.0}   # algorithmic bytes per particle-step of g2p2g: 2*4*C + 8
MATERIAL_NAMES = {0: "J_FLUID", 1: "FIXED_COROTATED", 2: "SAND", 3: "NACC"}
# CPU-arm sample of a workload: same geometry / grid / material / dt with the length scale reduced until the oracle port finishes
# a sub-step in about a second
CPU_SAMPLES = {"spheres40m": ("two_spheres", dict(domain_bits=9, radius=0.1645 / 2), "two elastic spheres (fixed-corotated), 512^3 grid, r=42 cells"),
               "spheres5m": ("two_spheres", dict(domain_bits=8, radius=0.1645 / 2), "two elastic spheres (fixed-corotated), 256^3 grid, r=21 cells"),
               "sand20m": ("sand_column", dict(domain_bits=9, size=(40, 60, 40)), "sand column (Drucker-Prager), 512^3 grid, 40x60x40 cells"),
               "fluid40m": ("fluid_dam", dict(domain_bits=10, size=(50, 32, 50)), "fluid dam, 1024^3 grid, 50x32x50 cells"),
               "mixed100m": ("mixed_materials", dict(domain_bits=10, edge=24), "mixed materials, 1024^3 grid, eight 24^3-cell bodies")}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (recipe in /opt/skills/guides/B200_PROFILING.md)."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc, self.thread = index, [], None, None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()
        t0 = time.time()
        while not self.rows and time.time() - t0 < 3.0:   # the first sample takes a few hundred ms: wait for it
            time.sleep(0.01)
        self.first = len(self.rows)

    def mark(self):
        """Samples from here on are 'under load' (warm-up, timed region, per-kernel timing pass)."""
        self.first = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows[max(getattr(self, "first", 0) - 1, 0):]:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def cpu_threads():
    """Threads for the CPU legs.  The oracle port stops scaling past 16 threads (measured on the 128-core B200 host with the
    0.63 M-particle sample: 8 -> 8.6, 16 -> 16.1, 32 -> 14.4, 64 -> 11.2, 128 -> 1.7 M particle-steps/s), so 16 is "all it can use"."""
    return max(1, min(os.cpu_count() or 1, 16))


def cpu_sample(workload_name):
    from claymore_b200 import scenes
    fn, kw, label = CPU_SAMPLES.get(workload_name, CPU_SAMPLES["spheres40m"])
    return getattr(scenes, fn)(**kw), label


def oracle_modules():
    """The CPU checker (tests/oracle_binding.py over oracle/libclaymore_oracle.so): cpu_baseline / --impl reference legs only."""
    t = os.path.join(ROOT, "tests")
    if t not in sys.path:
        sys.path.insert(0, t)
    import oracle_binding
    import scenes as test_scenes
    return oracle_binding, test_scenes


def time_cpu_port(scene, threads, seconds_budget=None, steps=None, warmup=1):
    """The oracle port on the host cores: (particle-steps/s in millions, particles, steps, seconds)."""
    from claymore_b200 import scenes
    ob, ts = oracle_modules()
    n = scenes.n_particles(scene)
    osim = ts.build_oracle(ob, scene, max_blocks=scenes.max_blocks_for(scene), threads=threads)
    osim.step(max(warmup, 1))
    t0 = time.perf_counter()
    done = 0
    while True:
        osim.step(1)
        done += 1
        el = time.perf_counter() - t0
        if (steps and done >= steps) or (seconds_budget and el >= seconds_budget):
            break
    osim.close()
    return n * done / el / 1e6, n, done, el


def run_reference(args):
    """--impl reference: the reference has no CPU implementation of this path (Projects/TaichiScripts/gmpm.py is a
    57-line stub, SURVEY.md 'Read this first' #4), so the arm times the oracle port (OpenMP) on the host cores, on a
    bounded sample of the arm's workload (same geometry, grid, material and dt; fewer particles)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from claymore_b200 import scenes
    cores = cpu_threads()
    scene, sample_label = cpu_sample(args.workload)
    n = scenes.n_particles(scene)
    v, _, steps, el = time_cpu_port(scene, cores, steps=args.steps, warmup=args.warmup)
    wl_label = workload_label(args.workload, args.gpus, args.scaling)
    sample = f"{sample_label}: {n} particles x {steps} sub-steps per timed run -- a bounded sample of the workload named in config.workload (same grid, material, dt)"
    out = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": el / steps * 1e3, "higher_is_better": True, "scaling": args.scaling if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl_label, "timed_sample": sample_label, "timed_particles": n, "note": "CPU port of the reference path (the reference ships no CPU implementation); per-particle throughput of the sample, not a run of the full workload"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


def workload_label(name, n_gpus, scaling):
    from claymore_b200 import scenes
    labels = {"spheres5m": "GMPM two elastic spheres (fixed-corotated), 256^3 grid, 5M particles",
              "spheres40m": "GMPM two elastic spheres (fixed-corotated), 512^3 grid, 40M particles",
              "sand20m": "GMPM sand column collapse (Drucker-Prager), 512^3 grid, 20M particles",
              "fluid40m": "weakly-compressible fluid dam break, 1024^3 grid, 40M particles",
              "mixed100m": "MGSP mixed materials (4 fluid + 2 sand + 2 fixed-corotated bodies), 1024^3 grid, 100M particles"}
    base = labels.get(name, name)
    if n_gpus > 1:
        if scaling == "weak":
            return f"MGSP two elastic spheres (fixed-corotated), {n_gpus}x5M particles, x-slab static partition (weak scaling)"
        return base.replace("GMPM", "MGSP") + f", static x-slab partition over {n_gpus} GPUs (strong scaling)"
    return base


def build_workload(name, n_gpus, scaling):
    from claymore_b200 import scenes
    if n_gpus > 1 and scaling == "weak":
        bits = 8 if n_gpus <= 2 else 9
        # same number of particles per rank: radius in cells scales with N^(1/3); keep the cell size of the chosen grid
        r_cells = 42.1 * n_gpus ** (1.0 / 3.0)
        r = r_cells / (1 << bits)
        gap = 0.05
        c0, c1 = 0.5 - gap / 2 - r, 0.5 + gap / 2 + r
        return scenes.two_spheres(domain_bits=bits, radius=r, centers=((c0, 0.5, 0.5), (c1, 0.5, 0.5)))
    return scenes.workload(name)[0]


def g2p2g_alg_bytes(per_model_counts, materials, pbc):
    """Algorithmic bytes of one sub-step's g2p2g work (SURVEY.md 8d): particles x B_p(material) + 2048 B per particle block and
    material launch."""
    by_mat = {}
    for n, m in zip(per_model_counts, materials):
        by_mat[m] = by_mat.get(m, 0) + n
    return sum(n * BYTES_BY_MATERIAL[m] for m, n in by_mat.items()) + pbc * BLOCK_BYTES_G2P2G * len(by_mat), len(by_mat)


DUMP_PARTICLES = 1 << 19    # particle states written by --dump-outputs, over all models
DUMP_BLOCKS = 1 << 13       # grid blocks written by --dump-outputs
DUMP_KEYS = 1 << 19         # block keys written by --dump-outputs


def dump_outputs(sim, outdir):
    """What a caller of the timed path receives after its last sub-step, as float32 / float64 .npy files (< 64 MB in all; larger
    outputs are represented by a fixed, seeded sample, so two builds run with the same arguments can be compared file by file):
      particles_<model>.npy  particle states (position, then the material's channels), sorted by position quantised to 1e-5
      grid_block_keys.npy    block coordinates of the sampled grid blocks, sorted by key
      grid_blocks.npy        their mass and momentum per cell [block][mass, mv_x, mv_y, mv_z][64 cells]
      active_keys.npy        all active block coordinates (particle, neighbour, exterior blocks), sorted by key
      stats.npy              particle / neighbour / exterior block counts, dt, next dt, max velocity, sub-steps taken"""
    from claymore_b200 import scenes
    os.makedirs(outdir, exist_ok=True)
    st = sim.stats()
    np.save(os.path.join(outdir, "stats.npy"), np.array([st.particle_block_count, st.neighbor_block_count, st.exterior_block_count,
                                                         st.dt, st.next_dt, st.max_vel, st.steps], np.float64))
    per_model = DUMP_PARTICLES // len(sim.counts)
    for m in range(len(sim.counts)):
        state = sim.particle_state(m)
        q = np.round(state[:, :3].astype(np.float64) * 1e5).astype(np.int64)   # positions lie in [0, 1]: 17 bits per axis
        order = np.argsort((q[:, 0] << 40) | (q[:, 1] << 20) | q[:, 2], kind="stable")
        if len(order) > per_model:
            order = order[np.sort(np.random.default_rng(m).choice(len(order), per_model, replace=False))]
        np.save(os.path.join(outdir, f"particles_{m}.npy"), state[order])
        del state
    keys = sim.active_keys()
    h = scenes.key_hash(keys)
    ko = np.argsort(h)
    if len(ko) > DUMP_KEYS:
        ko = ko[np.sort(np.random.default_rng(100).choice(len(ko), DUMP_KEYS, replace=False))]
    np.save(os.path.join(outdir, "active_keys.npy"), keys[ko].astype(np.float64))
    gh, gg = scenes.grid_by_key(keys, sim.grid())
    pick = np.arange(len(gh))
    if len(pick) > DUMP_BLOCKS:
        pick = np.sort(np.random.default_rng(101).choice(len(pick), DUMP_BLOCKS, replace=False))
    gkeys = np.stack([(gh[pick] >> 40) & 0xFFFFF, (gh[pick] >> 20) & 0xFFFFF, gh[pick] & 0xFFFFF], 1)
    np.save(os.path.join(outdir, "grid_block_keys.npy"), gkeys.astype(np.float64))
    np.save(os.path.join(outdir, "grid_blocks.npy"), gg[pick])


def device_timed(scene, args, stream, mb, max_ppc, clocks=None, dump_dir=None):
    """K sub-steps, CUDA events on the launching stream, graph replay (dump_dir: the state they leave is written there); then the
    same simulation's next K sub-steps as plain stream launches with an event pair around every g2p2g launch (roofline) and an
    event per phase."""
    import torch
    from claymore_b200 import scenes
    sim = scenes.build_engine(scene, dt=args.dt, max_blocks=mb, max_ppc=max_ppc, use_graph=not args.no_graph, stream=stream.cuda_stream, auto_grow=False)
    if clocks:
        clocks.mark()
    sim.step(args.warmup)
    sim.sync()
    st0 = sim.stats()
    assert st0.error == 0, f"engine error bits {st0.error} after warm-up"
    l0 = sim.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    sim.step(args.steps)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    launches = sim.launch_count - l0
    if dump_dir:
        dump_outputs(sim, dump_dir)
    sim.profile(True)
    sim.step(args.steps)
    g2p2g_ms, g2p2g_launches = sim.profile_read()
    phases_ms = {k: round(v / args.steps, 4) for k, v in sim.profile_phases().items()}
    sim.profile(False)
    st = sim.stats()
    assert st.error == 0, f"engine error bits {st.error}"
    sim.close()
    return dict(ms_total=ms_total, launches=launches, g2p2g_ms=g2p2g_ms, g2p2g_launches=g2p2g_launches, phases_ms=phases_ms, pbc=st.particle_block_count,
                nbc=st.neighbor_block_count, ebc=st.exterior_block_count)


def roofline_of(scene, res, steps, workload_name=None):
    per_model = [len(m["pos"]) for m in scene["models"]]
    mats = [m["material"] for m in scene["models"]]
    alg_step, n_mat = g2p2g_alg_bytes(per_model, mats, res["pbc"])
    launches_per_step = max(res["g2p2g_launches"], 1) / steps
    alg_bytes_per_launch = alg_step / launches_per_step
    avg_launch_s = res["g2p2g_ms"] / max(res["g2p2g_launches"], 1) * 1e-3
    peak, peak_kind = measured_peak_hbm()
    achieved = alg_bytes_per_launch / avg_launch_s / 1e9
    kern = "g2p2g_kernel<%s>" % "+".join(MATERIAL_NAMES[m] for m in sorted(set(mats)))
    r = {"bound": "hbm", "kernel": kern, "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
         "alg_bytes_per_launch": alg_bytes_per_launch, "avg_launch_ms": avg_launch_s * 1e3, "launches_timed": res["g2p2g_launches"],
         "share_of_step": (res["g2p2g_ms"] / steps) / (res["ms_total"] / steps),
         # secondary ceilings (SURVEY.md 8d): see profiles/ for the ncu figures these come from
         "secondary": read_secondary()}
    traffic_file = os.path.join(ROOT, "profiles", "g2p2g_traffic.json")
    if os.path.exists(traffic_file):
        try:
            with open(traffic_file) as f:
                r["traffic"] = json.load(f).get("by_workload", {}).get(workload_name, {}).get("dram_bytes_per_launch")
        except Exception:
            pass
    return r


def read_secondary():
    p = os.path.join(ROOT, "profiles", "g2p2g_secondary.json")
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return None


def time_ref_gpu(scene, steps, warmup, dt):
    """The reference's own GMPM kernels (unmodified, built for sm_100a by oracle/build_ref.sh) behind its host loop order, same
    scene, same GPU, same process: wall clock over `steps` sub-steps (its per-step syncs and D2H counter copies are part of what
    a user of the reference waits for; its prints and file output are not issued)."""
    t = os.path.join(ROOT, "tests")
    if t not in sys.path:
        sys.path.insert(0, t)
    import ref_gpu_binding as rg
    from claymore_b200 import scenes
    bits = scene["domain_bits"]
    mats = {m["material"] for m in scene["models"]}
    if not rg.available(bits) or len(mats) != 1 or next(iter(mats)) not in rg.CHANNELS:
        return None
    n = scenes.n_particles(scene)
    sim = rg.build_ref(scene, dt)
    sim.step(max(warmup, 1))
    ms = sim.time_steps(steps)
    pbc, nbc, ebc = sim.block_counts()
    sim.close()
    return {"value": n * steps / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms / steps, "steps": steps, "blocks": [pbc, nbc, ebc],
            "what": f"reference claymore GMPM kernels, sm_100a build of the unmodified sources (oracle/_ref/libclaymore_ref_gpu_d{bits}.so), reference host loop order, no prints / IO"}


def e2e_single(scene, args, stream, mb, max_ppc, repeats=2):
    """End to end through the public API with HOST buffers inside the timed region: upload of every model from pinned host memory
    (init_model), initial_setup, K sub-steps each followed by a device->host read of the step result (block counts, dt, max
    velocity), and the download of all particle positions.  The whole sequence is timed `repeats` times (each with a fresh
    simulator); the best run is reported and all of them are listed (host-side hiccups of a shared box show up as outliers)."""
    import torch
    import claymore_b200 as cb
    from claymore_b200 import scenes
    n_particles = scenes.n_particles(scene)
    dx = 1.0 / (1 << scene["domain_bits"])
    pinned = [torch.from_numpy(np.ascontiguousarray(m["pos"])).pin_memory() for m in scene["models"]]
    out_pinned = [torch.empty_like(p).pin_memory() for p in pinned]   # the caller's output buffers, reused frame after frame
    runs = []
    for _ in range(max(repeats, 1)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cfg = cb.Config(domain_bits=scene["domain_bits"], max_ppc=max_ppc)
        sim2 = cb.GmpmSimulator(dt=args.dt, fps=0, config=cfg, max_blocks=mb, use_graph=not args.no_graph, stream=stream.cuda_stream)
        for m, p in zip(scene["models"], pinned):
            mid = sim2.init_model(m["material"], p.numpy(), m["v0"])
            scenes.apply_material(sim2, mid, m["material"], dx)
        sim2.initial_setup()
        stats_bytes = 0
        for _ in range(args.steps):
            sim2.step(1)
            s = sim2.stats()
            stats_bytes += 76
        out_n = 0
        for i in range(len(scene["models"])):
            out_n += len(sim2.retrieve(i, out=out_pinned[i].numpy()))
        torch.cuda.synchronize()
        runs.append(time.perf_counter() - t0)
        assert out_n == n_particles and s.error == 0
        sim2.close()
    e2e_s = min(runs)
    return {"value": n_particles * args.steps / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": n_particles * 12 / args.steps,
            "d2h_bytes_per_step": n_particles * 12 / args.steps + stats_bytes / args.steps, "seconds": e2e_s, "seconds_all_runs": [round(r, 5) for r in runs],
            "note": "timed: simulator creation, init_model H2D from pinned host, initial_setup, K x (step + D2H stats), retrieve D2H of all positions; best of the listed runs"}


def run_b200(args):
    # rank 0 prints exactly one JSON line on stdout: NCCL's banner / debug lines (the box exports NCCL_DEBUG) go to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":  # this level alone printf()s a banner to stdout
        os.environ["NCCL_DEBUG"] = "WARN"
    import torch
    import torch.distributed as dist
    import claymore_b200 as cb
    from claymore_b200 import scenes

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 bench.py --gpus N ...")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cb.lib()  # fail loudly if the CUDA library is missing

    scene = build_workload(args.workload, world, args.scaling)
    label = workload_label(args.workload, world, args.scaling)
    max_ppc = args.max_ppc or (32 if args.workload.startswith("mixed") else 128)
    if world > 1:
        return bench_mgsp(args, scene, label, rank, world, local_rank, max_ppc)

    n_particles = scenes.n_particles(scene)
    mb = scenes.max_blocks_for(scene)
    stream = torch.cuda.Stream()  # the kernels are launched on this stream; the timing events are recorded on it too

    clocks = ClockSampler(local_rank)
    clocks.start()
    res = device_timed(scene, args, stream, mb, max_ppc, clocks, dump_dir=args.dump_outputs)
    clk = clocks.stop()
    value = n_particles * args.steps / (res["ms_total"] * 1e-3) / 1e6
    roofline = roofline_of(scene, res, args.steps, args.workload)
    e2e = e2e_single(scene, args, stream, mb, max_ppc)

    # ---- the reference's own kernels on the same scene, same GPU (the ">= 2x per GPU" denominator) ---------------------
    ref_gpu = None
    if not args.no_ref_gpu:
        cb.lib().cb200_trim_pool()   # hand the engine's pooled buffers back before the reference allocates its own
        torch.cuda.empty_cache()
        try:
            ref_gpu = time_ref_gpu(scene, min(args.steps, 30), args.warmup, args.dt)
        except Exception as e:  # the baseline leg must never take the bench line down
            ref_gpu = {"unavailable": f"{type(e).__name__}: {e}"}

    # ---- BASELINE configs[1] beside the headline scene (device-timed only) ------------------------------------------------
    configs1 = None
    if args.workload == "spheres40m" and not args.no_configs1:
        sc5, lab5 = scenes.workload("spheres5m")
        r5 = device_timed(sc5, args, stream, scenes.max_blocks_for(sc5), 128)
        n5 = scenes.n_particles(sc5)
        configs1 = {"workload": lab5, "value": n5 * args.steps / (r5["ms_total"] * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": r5["ms_total"] / args.steps,
                    "roofline_frac": roofline_of(sc5, r5, args.steps, "spheres5m")["frac"]}

    # ---- CPU baseline beside it: the oracle port on the host cores, bounded sample ---------------------------------------
    cpu = None
    if not args.no_cpu_baseline:
        cores = cpu_threads()
        sc, lab = cpu_sample(args.workload)
        v, n_s, steps_s, _ = time_cpu_port(sc, cores, seconds_budget=args.cpu_seconds)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": f"{lab}: {n_s} particles x {steps_s} sub-steps (~{args.cpu_seconds:.0f} s), oracle port (OpenMP)"}

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": res["ms_total"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": label, "particles": n_particles, "particle_blocks": res["pbc"], "blocks": [res["pbc"], res["nbc"], res["ebc"]], "dt": args.dt, "max_ppc": max_ppc,
                   "l2": "inputs larger than L2 (particle bins >= 500 MB)", "graph": not args.no_graph},
        "e2e": e2e, "gpu_launches": int(res["launches"]), "clocks": clk, "roofline": roofline, "cpu_baseline": cpu,
        "phases_ms": res["phases_ms"], "ref_gpu": ref_gpu, "configs1": configs1,
    }
    if ref_gpu and "value" in ref_gpu:
        out["vs_ref_gpu"] = value / ref_gpu["value"]
        out["vs_ref_gpu_e2e"] = e2e["value"] / ref_gpu["value"]
    print(json.dumps(out))


# ---------------------------------------------------------------------------------------------------------------------------
# N > 1: MGSP static particle partition, one process per GPU
# ---------------------------------------------------------------------------------------------------------------------------
def mgsp_parity(sim, part, scene, args, rank, world, mb_single, max_ppc, stream, steps_done):
    """Union of the shards against a single-GPU run of the same scene (rank 0), and owner agreement on shared grid blocks.
    Every rank contributes its active keys and grid blocks (mass + momentum of the grid the next sub-step starts from)."""
    import torch
    import torch.distributed as dist
    from claymore_b200 import scenes
    st = sim.stats()
    keys = sim.active_keys()[: st.neighbor_block_count]
    grid = sim.grid()                       # [nbc][4][64]
    counts = [len(sim.retrieve(i)) for i in range(len(part["models"]))]
    blob = dict(keys=keys, mass=grid[:, 0].sum(1).astype(np.float64), mom=grid[:, 1:].sum(2).astype(np.float64), cellmass=grid[:, 0], n=sum(counts), pbc=st.particle_block_count)
    gathered = [None] * world
    dist.all_gather_object(gathered, blob)
    if rank != 0:
        return None
    allk = np.concatenate([g["keys"] for g in gathered], 0)
    h = scenes.key_hash(allk)
    mass = np.concatenate([g["mass"] for g in gathered])
    mom = np.concatenate([g["mom"] for g in gathered], 0)
    cellmass = np.concatenate([g["cellmass"] for g in gathered], 0)
    # sort by key, and inside a key by decreasing block mass: the first copy of every key is the fullest one
    order = np.lexsort((-mass, h))
    hs = h[order]
    first = np.ones(len(hs), bool)
    first[1:] = hs[1:] != hs[:-1]
    grp = np.cumsum(first) - 1
    ref_mass = mass[order][first][grp]
    ref_mom = mom[order][first][grp]
    dup = ~first
    # Owner agreement.  Every owner of a shared grid block holds the sum of ALL ranks' contributions (the fused halo reduction),
    # with one protocol-inherent exception, shared with the reference's MGSP (mgsp_benchmark.cuh:421-467, 661-720): a block that
    # entered a rank's partition in the last sub-step was not yet tagged as shared when that sub-step's g2p2g ran, so that rank's
    # copy is still all zero for this one sub-step.  It is never read: a particle's next G2P stencil lies inside its previous
    # block's 2x2x2 neighbourhood, i.e. in blocks its rank already had.  Such copies are counted, every other copy must agree.
    fresh = dup & (mass[order] == 0.0) & (np.abs(mom[order]).sum(1) == 0.0) & (ref_mass != 0.0)
    chk = dup & ~fresh
    scale_m = max(float(np.abs(mass).max()), 1e-30)
    scale_p = max(float(np.abs(mom).max()), 1e-30)
    owner_mass_err = float(np.abs(mass[order] - ref_mass)[chk].max() / scale_m) if chk.any() else 0.0
    owner_mom_err = float(np.abs(mom[order] - ref_mom)[chk].max() / scale_p) if chk.any() else 0.0
    # blocks held by 3+ ranks exist when slabs are thinner than a block or the split is 2-D
    mult = np.bincount(grp)
    total_mass = float(mass[order][first].sum())
    total_mom = mom[order][first].sum(0)
    n_total = sum(g["n"] for g in gathered)
    mp = {}
    for m in scene["models"]:
        mp[m["material"]] = mp.get(m["material"], 0) + len(m["pos"])
    dx = 1.0 / (1 << scene["domain_bits"])
    expect_mass = sum(cnt * 1e3 * dx ** 3 / 8.0 for cnt in mp.values())
    out = {"particles_retrieved": int(n_total), "particles_expected": int(scenes.n_particles(scene)), "shared_blocks": int(dup.sum()), "max_owners_of_a_block": int(mult.max()),
           "shared_copies_checked": int(chk.sum()), "copies_new_on_their_rank_this_substep": int(fresh.sum()),
           "owner_mass_rel_err": owner_mass_err, "owner_momentum_rel_err": owner_mom_err, "grid_mass": total_mass, "grid_mass_expected": expect_mass,
           "grid_mass_rel_err": abs(total_mass - expect_mass) / expect_mass}
    ok = n_total == scenes.n_particles(scene) and owner_mass_err <= 1e-5 and owner_mom_err <= 1e-4 and out["grid_mass_rel_err"] <= 1e-5
    if not args.no_single_parity:
        # the same scene on ONE GPU (rank 0), same number of sub-steps
        single = scenes.build_engine(scene, dt=args.dt, max_blocks=mb_single, max_ppc=max_ppc, use_graph=True, stream=stream.cuda_stream, auto_grow=False)
        single.step(steps_done)
        sst = single.stats()
        skeys = single.active_keys()[: sst.neighbor_block_count]
        sgrid = single.grid()
        single.close()
        sh = scenes.key_hash(skeys)
        uniq = hs[first]
        so = np.argsort(sh)
        same_keys = len(uniq) == len(sh) and bool(np.array_equal(uniq, sh[so]))
        out["single_gpu_blocks"] = int(len(sh))
        out["union_blocks"] = int(len(uniq))
        out["key_sets_identical"] = same_keys
        out["key_set_symmetric_difference"] = int(len(np.setxor1d(uniq, sh)))
        smass, smom = sgrid[:, 0].sum(1).astype(np.float64), sgrid[:, 1:].sum(2).astype(np.float64)
        out["total_mass_rel_err_vs_single"] = abs(total_mass - smass.sum()) / smass.sum()
        out["total_momentum_err_vs_single"] = float(np.abs(total_mom - smom.sum(0)).max() / max(np.abs(smom).sum(0).max(), 1e-30))
        if same_keys:
            cm = cellmass[order][first]
            out["cell_mass_max_rel_err_vs_single"] = float(np.abs(cm - sgrid[so][:, 0]).max() / sgrid[:, 0].max())
            out["block_momentum_max_err_vs_single"] = float(np.abs(mom[order][first] - smom[so]).max() / np.abs(smom).max())
            ok = ok and out["cell_mass_max_rel_err_vs_single"] <= 1e-4 and out["block_momentum_max_err_vs_single"] <= 1e-3
        ok = ok and out["key_set_symmetric_difference"] <= max(2, len(sh) // 10000) and out["total_mass_rel_err_vs_single"] <= 1e-5
    out["ok"] = bool(ok)
    out["tolerances"] = "owners 1e-5 mass / 1e-4 momentum; grid mass 1e-5; vs single GPU: key sets identical (<= 0.01 % flips tolerated), cell mass 1e-4, block momentum 1e-3 of max"
    return out


def bench_mgsp(args, scene, label, rank, world, local_rank, max_ppc):
    """N>1 arm: max-over-ranks device time, rank 0 prints the JSON line."""
    import torch
    import torch.distributed as dist
    from claymore_b200 import mgsp, scenes

    part = mgsp.partition_scene_global(scene, rank, world) if args.scaling == "strong" else mgsp.partition_scene(scene, rank, world)
    n_local = scenes.n_particles(part)
    n_total = scenes.n_particles(scene)
    mb = mgsp.common_max_blocks(n_local, dist)   # the same on every rank: the inbox layout is computed from it on both sides
    mb_single = scenes.max_blocks_for(scene)
    stream = torch.cuda.Stream()
    sim = mgsp.build_rank_sim(part, rank, world, args.dt, mb, scenes.apply_material, stream=stream.cuda_stream, use_graph=not args.no_graph, max_ppc=max_ppc)
    mgsp.connect(sim, dist)
    sim.initial_setup()
    dist.barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
        clocks.mark()
    sim.step(args.warmup)
    sim.sync()
    assert sim.stats().error == 0, f"rank {rank}: engine error bits {sim.stats().error} after warm-up"
    l0 = sim.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier()
    torch.cuda.synchronize()
    e0.record(stream)
    sim.step(args.steps)
    e1.record(stream)
    torch.cuda.synchronize()
    dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    launches = sim.launch_count - l0
    sim.profile(True)
    sim.step(args.steps)
    phases = sim.profile_phases()
    g_ms, g_n = sim.profile_read()
    sim.profile(False)
    gathered = [None] * world
    dist.all_gather_object(gathered, {k: round(v / args.steps, 4) for k, v in phases.items()})
    clk = clocks.stop() if rank == 0 else None
    st = sim.stats()
    shared, halo_pb = sim.mgsp_halo_counts()
    err = torch.tensor([st.error], device="cuda")
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    assert int(err.item()) == 0, "engine error bits set on some rank"
    sizes = [None] * world
    dist.all_gather_object(sizes, (n_local, st.particle_block_count))

    parity = None
    if not args.no_parity:
        parity = mgsp_parity(sim, part, scene, args, rank, world, mb_single, max_ppc, stream, args.warmup + 2 * args.steps)
        dist.barrier()

    # end to end: upload from pinned host memory, setup, K x (step + D2H stats), download -- on every rank, max over ranks
    sim.close()
    pinned = [torch.from_numpy(m["pos"]).pin_memory() for m in part["models"]]
    out_pinned = [torch.empty_like(p).pin_memory() for p in pinned]
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    parts2 = dict(domain_bits=part["domain_bits"], models=[dict(material=m["material"], pos=p.numpy(), v0=m["v0"]) for m, p in zip(part["models"], pinned)])
    sim2 = mgsp.build_rank_sim(parts2, rank, world, args.dt, mb, scenes.apply_material, stream=stream.cuda_stream, use_graph=not args.no_graph, max_ppc=max_ppc)
    mgsp.connect(sim2, dist)
    sim2.initial_setup()
    for _ in range(args.steps):
        sim2.step(1)
        s2 = sim2.stats()
    got = sum(len(sim2.retrieve(i, out=out_pinned[i].numpy())) for i in range(len(part["models"])))
    torch.cuda.synchronize()
    t = torch.tensor([time.perf_counter() - t0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    assert got == n_local and s2.error == 0
    sim2.close()
    e2e_s = float(t.item())

    if rank == 0:
        per_model = [len(m["pos"]) for m in part["models"]]
        mats = [m["material"] for m in part["models"]]
        alg, n_mat = g2p2g_alg_bytes(per_model, mats, st.particle_block_count)   # per sub-step on this rank
        peak, kind = measured_peak_hbm()
        per_step_g2p2g_s = g_ms / args.steps * 1e-3
        achieved = alg / per_step_g2p2g_s / 1e9
        out = {
            "metric": METRIC, "value": n_total * args.steps / (ms_total * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": label, "particles": n_total, "particles_by_rank": [s[0] for s in sizes], "particle_blocks_by_rank": [s[1] for s in sizes], "dt": args.dt, "max_ppc": max_ppc,
                       "halo_blocks_shared_rank0": shared, "halo_particle_blocks_rank0": halo_pb, "l2": "inputs larger than L2", "graph": not args.no_graph, "phase_ms_per_step_by_rank": gathered,
                       "transport": "g2p2g bulk-add-reduces halo sums into the peers' grids over NVLink (CUDA-IPC peer memory); keys / max velocity through peer inboxes; NCCL (torch.distributed) for rendezvous and timing only"},
            "e2e": {"value": n_total * args.steps / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": n_local * 12 / args.steps, "d2h_bytes_per_step": n_local * 12 / args.steps + 76, "seconds": e2e_s},
            "gpu_launches": int(launches), "clocks": clk,
            "roofline": {"bound": "hbm", "kernel": "g2p2g_kernel (rank 0)", "achieved": achieved, "peak": peak, "peak_kind": kind, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": None, "alg_bytes_per_launch": alg / max(g_n / args.steps, 1), "launches_timed": g_n},
            "cpu_baseline": None, "parity": parity,
        }
        print(json.dumps(out))
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="spheres40m")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--dt", type=float, default=1e-4)
    ap.add_argument("--max-ppc", type=int, default=0)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--no-configs1", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-single-parity", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the state the timed sub-steps leave as .npy files into DIR (--gpus 1)")
    args = ap.parse_args()
    if args.dump_outputs and (args.gpus != 1 or args.impl != "b200"):
        ap.error("--dump-outputs needs --gpus 1 and --impl b200")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
