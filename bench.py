#!/usr/bin/env python
"""bench.py — particle-steps/s of the salva3d DFSPH step path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            native arm (this repo's CUDA engine)
  python bench.py --impl reference --gpus N --steps K ...   reference arm: the CPU restatement of salva's own
                                                            algorithm (oracle/, kind "port": the Rust reference
                                                            cannot be built here) on the box's host cores
  python bench.py --gpus 1 --steps K --dump-outputs DIR     also writes the fluid state after the last timed step as .npy
                                                            files, so that two builds can be compared on identical inputs

One "step" = one LiquidWorld::step (liquid_world.rs:62) of the whole world.
Workload: N = 1 -> BASELINE.json configs[2], C3 (216^3 = 10 077 696 particles, DFSPH + Akinci2013 surface tension:
the roofline-capture configuration); N > 1 -> configs[3], C4 sliced at 4M particles per GPU (64N x 250 x 250 block,
DFSPH, no extra force, 1-D x-slabs; N = 8 is the full 512 x 250 x 250 = 32M scene).  `--config c1|c2|c3|c4|c5` overrides.
Prints ONE JSON line on rank 0.

Timing: device time of every step from CUDA events recorded on the engine's own stream (sph_step_stats.step_ms),
W >= 3 warm-up steps, working set (particle state + neighbour lists, GBs) far larger than the 126 MB L2.
Before the timed region a >= 262k-particle copy of the workload is stepped on the GPU and on the CPU oracle with
forced iteration counts and compared (`parity` block; the run FAILS, rc 3, when it is out of tolerance); with N > 1 the
N-rank slab world is also compared with a 1-rank world of the same scene by particle id.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "particle-steps/s (DFSPH 3D)"
UNIT = "particle-steps/s"

# SURVEY.md §8(d) algorithmic bytes per particle per launch (compulsory-traffic model)
BYTES = dict(grid=136, density_alpha=24, divergence_eval=40, divergence_update=52, fold=64, xsph=52, artificial=52,
             akinci=104, integrate=64, predict_density=44, pressure_update=52, positions=64)
FORCE_NAMES = {0: "XSPHViscosity", 1: "ArtificialViscosity", 2: "Akinci2013SurfaceTension", 3: "Becker2009Elasticity",
               4: "He2014SurfaceTension", 5: "WCSPHSurfaceTension", 6: "DFSPHViscosity"}
PER_GPU_NX = 64  # C4 slices: 64 x 250 x 250 = 4M particles per GPU


def peaks():
    # Roofline denominator: median of 50 device-to-device copies of 4 GiB (bytes read + written), timed with CUDA events on an
    # NVIDIA B200 at its 1000 W power limit (SM clock max 1965 MHz).  Kept here so every run divides by the same measured number.
    return 6531.0, "measured: 4 GiB device-to-device copy, read + write, median of 50, NVIDIA B200 at 1000 W"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device=0):
        self.device = device
        self.proc = None
        self.lines = []
        self.t_mark = 0

    def mark(self):
        """Samples taken from here on belong to the timed region."""
        self.t_mark = len(self.lines)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = self.lines[self.t_mark:] if len(self.lines) - self.t_mark >= 2 else self.lines
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- workloads -------------------------------------------------------------------------------------------------------
def default_config(world_size):
    return "c3" if world_size == 1 else "c4"


def scene_dims(cfg, n, world_size):
    """Lattice dimensions (nx, ny, nz) of the block of `cfg`; n overrides the edge (tests / bounded CPU samples)."""
    if cfg == "c2":
        e = n or 100
        return e, e, e
    if cfg == "c3":
        e = n or 216
        return e, e, e
    if cfg == "c4":
        if n:
            return n * world_size, n, n
        return PER_GPU_NX * world_size, 250, 250
    return None


def scene_fn(cfg):
    from salva_b200 import scenes
    return {"c2": lambda nx, ny, nz, **kw: scenes._dam_break(nx, ny, nz, 0.025, 1.0e-3, [scenes.xsph_viscosity(0.5, 0.0)], name="C2", **kw),
            "c3": lambda nx, ny, nz, **kw: scenes._dam_break(nx, ny, nz, 0.025, 1.0e-3, [scenes.akinci2013_surface_tension(1.0, 0.0)], name="C3", **kw),
            "c4": lambda nx, ny, nz, **kw: scenes._dam_break(nx, ny, nz, 0.025, 1.0e-3, [], name="C4", tank_x_factor=1.25, **kw)}[cfg]


def build_scene(cfg, n=0, world_size=1, rank=None, **kw):
    """Whole scene (rank None) or rank's slab of it."""
    from salva_b200 import scenes
    if cfg == "c1":
        return scenes.scene_c1()
    if cfg == "c5":
        return scenes.scene_c5(n or 100)
    nx, ny, nz = scene_dims(cfg, n, world_size)
    fn = scene_fn(cfg)
    if rank is None or world_size == 1:
        return fn(nx, ny, nz, **kw)
    return scenes.slab_scene(lambda **k2: fn(nx, ny, nz, **k2), rank, world_size, nx, **kw)


def workload_name(cfg, n, world_size):
    base = {"c1": "C1 examples3d/basic3.rs 3375 particles, DFSPH + ArtificialViscosity",
            "c2": "C2 1M-particle cube dam-break, DFSPH + XSPH viscosity",
            "c3": "C3 10M particles (216^3) DFSPH + Akinci2013 surface tension, 1 GPU",
            "c4": "C4 DFSPH dam-break, 1-D x-slabs, 4M particles per GPU (64N x 250 x 250; N = 8 is the 32M scene)",
            "c5": "C5 2M particles IISPH + ArtificialViscosity + Becker2009, 2 fluids"}[cfg]
    return base + (" [lattice edge override %d]" % n if n else "")


def scene_counts(cfg, n, world_size):
    """(fluid particles, boundary particles) of the WHOLE workload without generating the fluid block."""
    from salva_b200 import scenes
    if cfg in ("c1", "c5"):
        sc = build_scene(cfg, n)
        return sum(len(f["positions"]) for f in sc["fluids"]), sum(len(b["positions"]) for b in sc["boundaries"])
    nx, ny, nz = scene_dims(cfg, n, world_size)
    tank = scene_fn(cfg)(nx, ny, nz, x_range=(0, 0))["boundaries"][0]["positions"]
    return nx * ny * nz, len(tank)


def static_config(cfg, n, world_size):
    """The part of `config` both arms print identically (the reference arm times a bounded SAMPLE of this workload)."""
    from salva_b200 import scenes  # noqa: F401
    nf, nb = scene_counts(cfg, n, world_size)
    sc = build_scene(cfg, 4 if cfg in ("c2", "c3", "c4") else n, world_size) if cfg not in ("c1", "c5") else build_scene(cfg, n)
    forces = [FORCE_NAMES[k] for f in sc["fluids"] for k, _ in f.get("forces", [])]
    return {"workload": workload_name(cfg, n, world_size), "fluid_particles_total": int(nf), "boundary_particles": int(nb),
            "solver": "DFSPH" if sc["solver"] == 0 else "IISPH", "forces": forces, "dt": sc["dt"],
            "particle_radius": sc["particle_radius"], "n_gpus": world_size,
            "l2": "inputs larger than L2: particle state + neighbour lists of one step are ~%.1f GB per GPU (L2 = 126 MB)"
                  % (nf / world_size * (16 * 8 + 4 * 10 + 48 * 4) / 1e9)}


# ---- CPU oracle (test infrastructure: parity checker + timed baseline) ---------------------------------------------
def best_oracle_threads(sc):
    """The port is timed with whichever host thread count is FASTEST on this box (oversubscribed hyper-threads
    or cgroup-limited cores make `all threads` several times slower: profiles/r1_oracle_thread_scaling.json)."""
    from oracle.oracle import OracleWorld
    from salva_b200 import scenes
    ncpu = os.cpu_count() or 1
    cands = sorted({t for t in (8, 16, 32, 64, ncpu) if t <= ncpu})
    best, best_t = None, None
    for th in cands:
        w = OracleWorld(sc["particle_radius"], sc["smoothing_factor"], solver=sc["solver"], sort_contacts=False, num_threads=th)
        scenes.populate(w, sc)
        w.step(sc["dt"], sc["gravity"])
        t0 = time.perf_counter()
        w.step(sc["dt"], sc["gravity"])
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = th, dt
    return best


def run_oracle(sc, steps, warmup, threads=0):
    """CPU restatement of the reference algorithm (oracle/, test infrastructure) timed on host cores."""
    from oracle.oracle import OracleWorld
    from salva_b200 import scenes
    if threads <= 0:
        small = dict(sc)
        threads = best_oracle_threads(sc) if sum(len(f["positions"]) for f in sc["fluids"]) <= 300000 else 0
        del small
    if threads <= 0:
        # large sample: probe the thread count on a 64^3 block of the same generator instead of on the sample itself
        threads = min(os.cpu_count() or 1, 32)
    w = OracleWorld(sc["particle_radius"], sc["smoothing_factor"], solver=sc["solver"], sort_contacts=False, num_threads=threads)
    scenes.populate(w, sc)
    for _ in range(warmup):
        w.step(sc["dt"], sc["gravity"])
    t0 = time.perf_counter()
    iters = []
    for _ in range(steps):
        w.step(sc["dt"], sc["gravity"])
        st = w.stats()
        iters.append((st["n_divergence_iter"], st["n_pressure_iter"]))
    dt = time.perf_counter() - t0
    nf = sum(len(f["positions"]) for f in sc["fluids"])
    st = w.stats()
    run_oracle.last_stages = {k: st[k] for k in st if k.endswith("_ms")}  # stage times of the LAST step (Counters-like, SURVEY 8d)
    return nf * steps / dt, dt / steps * 1e3, st["threads"], iters


def host_info():
    model = "unknown"
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"nproc": os.cpu_count() or 1, "cpu_model": model}


def cpu_extras(cfg):
    """Host description, per-stage ms of the last timed step of the port, and the same port on ONE thread (64^3 probe block)."""
    out = dict(host_info())
    out["stages_ms_last_step"] = {k: round(v, 3) for k, v in getattr(run_oracle, "last_stages", {}).items()}
    try:
        probe = build_scene(cfg, 64, 1) if cfg in ("c2", "c3", "c4") else build_scene(cfg, 0, 1)
        v1, ms1, _, _ = run_oracle(probe, 1, 1, 1)
        out["single_thread"] = {"value": v1, "unit": UNIT, "particles": sum(len(f["positions"]) for f in probe["fluids"]), "ms_per_step": ms1}
    except Exception as e:  # the extras never break the line
        out["single_thread"] = {"error": str(e)[:100]}
    return out


def cpu_sample_edge(cfg, n, ref_n):
    """Lattice edge of the bounded CPU sample: the whole workload when it is <= ~1M particles (C1, C2), else a 100^3
    block of the same generator (C3 / C4: the oracle needs ~1.6 KB per particle of cached contacts and ~0.5 s per
    million particle-steps, so 10M+ particles do not fit a few-minute run)."""
    if ref_n:
        return ref_n
    if cfg == "c2":
        return n or 100
    if cfg in ("c3", "c4"):
        return min(n or 100, 100)
    return n


def reference_arm(args, rank, world_size):
    """--impl reference: the reference's own CPU algorithm on the box's host cores (oracle port)."""
    if rank != 0:
        return
    cfg = args.config or default_config(world_size)
    edge = cpu_sample_edge(cfg, args.n, args.ref_n)
    sc = build_scene(cfg, edge, 1)
    nf = sum(len(f["positions"]) for f in sc["fluids"])
    probe = build_scene(cfg, min(edge or 64, 64), 1) if cfg in ("c2", "c3", "c4") else sc
    threads = best_oracle_threads(probe)
    value, ms, threads, iters = run_oracle(sc, args.steps, args.warmup, threads)
    extras = cpu_extras(cfg)
    conf = static_config(cfg, args.n, world_size)
    sample = ("%s generator at %d fluid particles (%s), %d host threads (fastest of 8..nproc on a 64^3 probe), %d+%d steps, %.0f ms/step"
              % (cfg.upper(), nf, "the whole workload" if nf == conf["fluid_particles_total"] else "bounded sample of the workload", threads,
                 args.warmup, args.steps, ms))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": conf,
            "sample_particles": nf, "iterations_last_step": list(iters[-1]) if iters else None,
            "cpu_baseline": dict({"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample}, **extras),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---- parity block ------------------------------------------------------------------------------------------------------
PARITY_TOL = {"max_dx_over_h": 1.0e-3, "max_rel_rho": 1.0e-5, "max_dv_over_h_dt": 1.0e-3}


def parity_vs_oracle(cfg, device, edge=64, steps=3):
    """GPU (through the C ABI) vs the CPU oracle on an edge^3 (>= 262k at 64) copy of the bench workload, started 7 %
    compressed so the pressure terms are exercised, forced iteration counts (2 divergence, 3 pressure updates)."""
    from oracle.oracle import OracleWorld
    from salva_b200 import DFSPHSolver, LiquidWorld, scenes
    sc = build_scene(cfg if cfg in ("c2", "c3", "c4") else "c3", edge, 1, compress=0.93, amplitude=0.3)
    gpu = LiquidWorld(DFSPHSolver(), particle_radius=sc["particle_radius"], smoothing_factor=sc["smoothing_factor"], device=device)
    cpu = OracleWorld(sc["particle_radius"], sc["smoothing_factor"], solver=0, num_threads=min(os.cpu_count() or 1, 32))
    (fg,), _ = scenes.populate(gpu, sc)
    (fc,), _ = scenes.populate(cpu, sc)
    for w in (gpu, cpu):
        w.force_iterations(2, 3)
    t0 = time.perf_counter()
    contacts_equal = None
    for k in range(steps):
        gpu.step(sc["dt"], sc["gravity"])
        cpu.step(sc["dt"], sc["gravity"])
        if k == 0:
            # exact comparison on IDENTICAL inputs (the first step's positions); from the second step on the two trajectories
            # differ by ~1e-6 h and a few of the 9M pairs sit that close to the cutoff, so later counts may differ legitimately
            contacts_equal = bool(np.array_equal(gpu.debug(fg, "num_fluid_contacts"), cpu.debug(fc, "num_fluid_contacts")) and
                                  np.array_equal(gpu.debug(fg, "num_boundary_contacts"), cpu.debug(fc, "num_boundary_contacts")))
    pg, vg = gpu.read_fluid(fg)
    pc, vc = cpu.read_fluid(fc)
    h = float(gpu.h)
    rg, rc = gpu.debug(fg, "density"), cpu.debug(fc, "density")
    res = {"n": int(len(pg)), "steps": steps, "forced_iterations": [2, 3], "scene": "%s generator, edge %d, lattice 0.93-compressed" % (cfg.upper(), edge),
           "contacts_equal": contacts_equal,
           "contact_count_mismatches_last_step": int((gpu.debug(fg, "num_fluid_contacts") != cpu.debug(fc, "num_fluid_contacts")).sum()),
           "max_dx_over_h": float(np.abs(pg - pc).max() / h),
           "max_dv_over_h_dt": float(np.abs(vg - vc).max() / (h / sc["dt"])),
           "max_rel_rho": float(np.abs(rg - rc).max() / np.abs(rc).max()),
           "tolerance": PARITY_TOL, "seconds": round(time.perf_counter() - t0, 2)}
    res["ok"] = bool(res["contacts_equal"] and res["max_dx_over_h"] <= PARITY_TOL["max_dx_over_h"] and
                     res["max_rel_rho"] <= PARITY_TOL["max_rel_rho"] and res["max_dv_over_h_dt"] <= PARITY_TOL["max_dv_over_h_dt"])
    gpu.close()
    return res


def parity_slab_vs_single(cfg, rank, world_size, local_rank, uid_fn, steps=6):
    """N-rank slab world vs a 1-rank world of the same scene (rank 0's GPU), matched by particle id."""
    import torch.distributed as dist
    from salva_b200 import DFSPHSolver, LiquidWorld, scenes, slab
    nx = 8 * world_size + 8
    whole = scene_fn(cfg)(nx, 24, 20, compress=0.93, amplitude=0.3)
    rng = np.random.default_rng(5)
    p = whole["fluids"][0]["positions"]
    vel = rng.normal(0, 0.2, p.shape).astype(np.float32)
    vel[:, 0] += np.where(p[:, 0] < p[:, 0].mean(), 1.0, -1.0).astype(np.float32)  # push particles across the planes
    whole["fluids"][0]["velocities"] = vel
    w = LiquidWorld(DFSPHSolver(), particle_radius=whole["particle_radius"], device=local_rank)
    fh, _ = slab.populate_slab(w, whole, rank, world_size, uid_fn())
    w.force_iterations(2, 3)
    migrated = 0
    for _ in range(steps):
        w.step(whole["dt"], whole["gravity"])
        migrated += w.stats()["n_migrated"]
    pp, vv = w.read_fluid(fh[0])
    ids = w.read_ids(fh[0])
    gathered = [None] * world_size
    dist.gather_object(dict(ids=ids, p=pp, v=vv, migrated=migrated), gathered if rank == 0 else None, dst=0)
    res = None
    if rank == 0:
        ids = np.concatenate([g["ids"] for g in gathered])
        pp = np.concatenate([g["p"] for g in gathered])
        order = np.argsort(ids)
        ref = LiquidWorld(DFSPHSolver(), particle_radius=whole["particle_radius"], device=local_rank)
        (fr,), _ = scenes.populate(ref, whole)
        ref.force_iterations(2, 3)
        for _ in range(steps):
            ref.step(whole["dt"], whole["gravity"])
        pr, _ = ref.read_fluid(fr)
        h = float(ref.h)
        ok_ids = len(ids) == len(pr) and len(np.unique(ids)) == len(ids)
        res = {"n": int(len(pr)), "ranks": world_size, "steps": steps, "ids_complete": bool(ok_ids),
               "migrated": int(sum(g["migrated"] for g in gathered)),
               "max_dx_over_h": float(np.abs(pp[order] - pr).max() / h) if ok_ids else None}
        res["ok"] = bool(ok_ids and res["max_dx_over_h"] <= PARITY_TOL["max_dx_over_h"])
        ref.close()
    w.close()
    return res


# ---- native arm --------------------------------------------------------------------------------------------------------
def timed_steps(world, sc, steps, barrier):
    acc, launches, iters = {}, 0, []
    st = {}
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        world.step(sc["dt"], sc["gravity"])
        st = world.stats()
        for k, v in st.items():
            if k.endswith("_ms"):
                acc[k] = acc.get(k, 0.0) + v
        for k in ("n_pressure_eval", "n_pressure_iter", "n_divergence_eval", "n_divergence_iter"):
            acc[k] = acc.get(k, 0) + st[k]
        launches += st["kernel_launches"]
        iters.append((st["n_divergence_iter"], st["n_pressure_iter"]))
        timed_steps.per_step.append((round(st["step_ms"], 3), round(st["grid_ms"], 3)))
    barrier()
    wall = time.perf_counter() - t0
    return acc, launches, iters, wall, st


timed_steps.per_step = []   # (step_ms, grid_ms) of every timed step on this rank: a one-off stall shows up here, not in the mean

DUMP_MAX_PARTICLES = 1 << 21   # positions + velocities in f32: 48 MB, within the 64 MB that --dump-outputs may write


def dump_outputs(world, fh, out_dir):
    """What a caller of LiquidWorld::step receives after the last timed step: positions and velocities of every fluid in original
    particle order, as out_dir/fluid<k>_{positions,velocities}.npy (f32).  Above DUMP_MAX_PARTICLES in all, fluid k keeps a fixed
    sample (sorted indices drawn with seed k) of its share of that budget, so that two builds given the same arguments write the
    same particles and can be compared array for array."""
    counts = [world.num_particles(f) for f in fh]
    total = sum(counts)
    os.makedirs(out_dir, exist_ok=True)
    for k, (f, n) in enumerate(zip(fh, counts)):
        p, v = world.read_fluid(f)
        if total > DUMP_MAX_PARTICLES:
            keep = np.sort(np.random.default_rng(k).choice(n, DUMP_MAX_PARTICLES * n // total, replace=False))
            p, v = p[keep], v[keep]
        np.save(os.path.join(out_dir, "fluid%d_positions.npy" % k), p)
        np.save(os.path.join(out_dir, "fluid%d_velocities.npy" % k), v)


def pick_grid_order(args, cfg, world_size):
    """Engine option Consts::xysub (SALVA_B200_XYSUB): 'rows' sorts the particles into (h/2 x h/2) columns with z running fastest, so
    that the lanes of a warp gather consecutive records (profiles/r2_l1tex_wavefront_model.md).  It changes the order of every f32 sum
    (not the contact sets), so it is only ever used after THIS run has checked it: both orders run as short subprocess probes that
    carry the same parity block as the real line, and 'rows' is kept only if its parity passes and it is faster in the timed
    free-fall steps without being slower in the settled block.  Anything going wrong in a probe => the default order."""
    info = {"chosen": "h", "mode": args.grid_order}
    if args.grid_order in ("h", "rows"):
        info["chosen"] = args.grid_order
        return info
    if world_size != 1 or args.backend != 0 or cfg not in ("c2", "c3", "c4") or args.probe:
        info["mode"] = "fixed (auto applies to one-GPU DFSPH dam-break configs)"
        return info
    import subprocess
    probes = {}
    for name in ("h", "rows"):
        cmd = [sys.executable, os.path.abspath(__file__), "--config", cfg, "--gpus", "1", "--steps", "5", "--warmup", "3", "--no-cpu", "--probe",
               "--grid-order", name, "--parity-n", str(args.parity_n)]
        if args.n:
            cmd += ["--n", str(args.n)]
        if args.no_settled:
            cmd += ["--no-settled"]
        try:
            t0 = time.perf_counter()
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=150)
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            d = json.loads(line[-1]) if line else None
            if r.returncode != 0 or d is None:
                probes[name] = {"error": "rc %d: %s" % (r.returncode, (r.stderr or "")[-200:].replace("\n", " | "))}
            else:
                probes[name] = {"ms_per_step": d["ms_per_step"], "parity_ok": bool((d.get("parity") or {}).get("ok")),
                                "pair_ms": d["roofline"]["ms_per_launch_pair"], "neighbors_ms": d["phases"].get("neighbors_ms"),
                                "grid_ms": d["phases"].get("grid_ms"),
                                "settled_ms_per_step": (d.get("settled") or {}).get("ms_per_step"),
                                "settled_error": (d.get("settled") or {}).get("error"), "seconds": round(time.perf_counter() - t0, 1)}
        except Exception as e:  # timeout, unparsable output, ...
            probes[name] = {"error": str(e)[:200]}
    info["probes"] = probes
    h, rows = probes.get("h", {}), probes.get("rows", {})
    ok = ("error" not in h and "error" not in rows and rows.get("parity_ok") and h.get("parity_ok") and
          not rows.get("settled_error") and rows["ms_per_step"] < 0.97 * h["ms_per_step"] and
          (rows.get("settled_ms_per_step") is None or h.get("settled_ms_per_step") is None or
           rows["settled_ms_per_step"] <= 1.02 * h["settled_ms_per_step"]))
    info["chosen"] = "rows" if ok else "h"
    return info


def native_arm(args, rank, world_size):
    import torch
    import torch.distributed as dist
    from salva_b200 import DFSPHSolver, IISPHSolver, LiquidWorld, scenes, slab
    from salva_b200.liquid_world import nccl_unique_id

    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world_size > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world_size > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def allsum(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world_size > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(x) for x in t]

    cfg = args.config or default_config(world_size)
    if world_size > 1 and cfg not in ("c2", "c3", "c4"):
        raise SystemExit("multi-GPU runs need a dam-break config (c2, c3 or c4)")
    uid_fn = (lambda: slab.broadcast_unique_id(nccl_unique_id, rank, device=dev)) if world_size > 1 else None
    grid_order = pick_grid_order(args, cfg, world_size)
    os.environ["SALVA_B200_XYSUB"] = "2" if grid_order["chosen"] == "rows" else "1"   # read by every world this process creates

    # ---- parity before anything is timed -----------------------------------------------------------------------------
    parity = None
    if not args.no_parity:
        parity = {}
        if rank == 0:
            parity = parity_vs_oracle(cfg, local_rank, edge=args.parity_n)
        if world_size > 1:
            sres = parity_slab_vs_single(cfg, rank, world_size, local_rank, uid_fn)
            if rank == 0:
                parity["slab_vs_single_gpu"] = sres
                parity["ok"] = bool(parity["ok"] and sres["ok"])

    def make_world(**kw):
        sc = build_scene(cfg, args.n, world_size, rank if world_size > 1 else None, **kw)
        solver = DFSPHSolver() if sc["solver"] == 0 else IISPHSolver()
        world = LiquidWorld(solver, particle_radius=sc["particle_radius"], smoothing_factor=sc["smoothing_factor"],
                            device=local_rank, deterministic=not args.fast_sort, gather_backend=args.backend)
        if world_size > 1:
            fh, _ = slab.populate_slab(world, sc, rank, world_size, uid_fn())
        else:
            fh, _ = scenes.populate(world, sc)
        return sc, world, fh

    sc, world, fh = make_world()
    nf_local = sum(len(f["positions"]) for f in sc["fluids"])
    nf = int(allsum([nf_local])[0]) if world_size > 1 else nf_local
    nb = sum(len(b["positions"]) for b in sc["boundaries"])
    if args.force_iters:
        world.force_iterations(*args.force_iters)
    warm = max(args.warmup, 3)
    sampler = ClockSampler(local_rank)
    sampler.start()  # nvidia-smi needs ~0.2 s to emit its first sample: start it before the warm-up steps
    for _ in range(warm):
        world.step(sc["dt"], sc["gravity"])

    # ---- timed region: device-resident inputs, CUDA-event time of every step -------------------------------------
    sampler.mark()
    timed_steps.per_step = []
    acc, launches, iters, wall, st = timed_steps(world, sc, args.steps, barrier)
    per_step = list(timed_steps.per_step)
    clocks = sampler.stop()
    dev_s, wall = allmax([acc["step_ms"] * 1e-3, wall])
    value = nf * args.steps / dev_s
    if args.dump_outputs:
        dump_outputs(world, fh, args.dump_outputs)   # before the e2e loop below steps the same world again

    # ---- e2e: the reference-facing call sequence with HOST buffers, copies inside the timed region ----------------
    f0 = fh[0]
    n0 = world.num_particles(f0)
    cap0 = int(n0 * 1.25) + 1024  # slab worlds gain / lose particles through migration
    hp_all = torch.empty((cap0, 3), dtype=torch.float32, pin_memory=True).numpy()
    hv_all = torch.empty((cap0, 3), dtype=torch.float32, pin_memory=True).numpy()
    world.read_fluid(f0, hp_all[:n0], hv_all[:n0])
    e2e_steps = 1 if args.probe else max(3, min(args.steps, 10))
    h2d = d2h = 0
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        world.write_fluid(f0, hp_all[:n0], hv_all[:n0])   # host edits of fluid.positions / velocities go in
        h2d += n0 * 24
        world.step(sc["dt"], sc["gravity"])               # LiquidWorld::step
        n0 = world.num_particles(f0)
        world.read_fluid(f0, hp_all[:n0], hv_all[:n0])    # results come back in original index order
        d2h += n0 * 24
    barrier()
    e2e_wall = allmax([time.perf_counter() - t0])[0]
    e2e_value = nf * e2e_steps / e2e_wall
    h2d, d2h = allsum([h2d / e2e_steps, d2h / e2e_steps])  # all ranks together, per step
    world.close()
    del hp_all, hv_all

    # ---- second measurement: the Jacobi loops iterate.  Start from a 0.92-compressed lattice (+2.7 % density): for the next
    # ~8 steps the divergence loop runs 4-6 updates per step while the block relaxes (probed on the oracle; a stronger
    # compression, 0.90, blows the block apart at 100 m/s through the tank walls, which is neither a meaningful regime nor kind
    # to a dense cell grid).  One GPU only: the driver's scaling runs stay as short (and as safe) as possible.
    settled = None
    if not args.no_settled and world_size == 1:
      try:
        sc2, w2, _ = make_world(compress=0.92)
        w2.step(sc2["dt"], sc2["gravity"])   # the first step only sees dt = 0 quantities (timestep_manager.rs:29-30)
        k2 = 8
        acc2, _, iters2, wall2, st2 = timed_steps(w2, sc2, k2, barrier)
        dev2 = allmax([acc2["step_ms"] * 1e-3])[0]
        settled = {"what": "same workload started from a 0.92-compressed lattice (+2.7 %% density): 1 warm-up + %d timed steps while the block relaxes" % k2,
                   "value": nf * k2 / dev2, "unit": UNIT, "ms_per_step": dev2 / k2 * 1e3,
                   "iterations_per_step_mean": [float(np.mean([i[0] for i in iters2])), float(np.mean([i[1] for i in iters2]))],
                   "pressure_pair_ms": (acc2["predict_density_ms"] / max(acc2["n_pressure_eval"], 1) +
                                        acc2["pressure_update_ms"] / max(acc2["n_pressure_iter"], 1)),
                   "divergence_pair_ms": (acc2["divergence_eval_ms"] / max(acc2["n_divergence_eval"] - k2, 1) +
                                          acc2["divergence_update_ms"] / max(acc2["n_divergence_iter"], 1)),
                   "wall_ms_per_step": wall2 / k2 * 1e3, "max_neighbors": st2.get("max_neighbors"), "grid_dims": st2.get("grid_dims"),
                   "phases": {k: acc2[k] / k2 for k in sorted(acc2) if k.endswith("_ms")}}
        w2.close()
      except Exception as e:   # the second measurement never costs the line
        settled = {"error": str(e)[:300]}

    # ---- N > 1: the same per-GPU slice on ONE GPU (rank 0, the others wait), so the line carries its own weak-scaling reference
    slice_ref = None
    if world_size > 1 and not args.no_slice_ref:
        if rank == 0:
            nx, ny, nz = scene_dims(cfg, args.n, world_size)
            one = scene_fn(cfg)(nx // world_size, ny, nz)
            w1 = LiquidWorld(DFSPHSolver(), particle_radius=one["particle_radius"], smoothing_factor=one["smoothing_factor"], device=local_rank,
                             deterministic=not args.fast_sort)
            scenes.populate(w1, one)
            for _ in range(3):
                w1.step(one["dt"], one["gravity"])
            k1 = max(3, min(args.steps, 10))
            ms1 = 0.0
            for _ in range(k1):
                w1.step(one["dt"], one["gravity"])
                ms1 += w1.stats()["step_ms"]
            n1 = len(one["fluids"][0]["positions"])
            slice_ref = {"what": "the %d-particle slice one rank owns, stepped alone on one GPU (no slabs), %d steps" % (n1, k1),
                         "value": n1 * k1 / (ms1 * 1e-3), "unit": UNIT, "ms_per_step": ms1 / k1}
            w1.close()
        barrier()
    if rank != 0:
        return 0
    peak, peak_src = peaks()
    # ---- roofline of the pressure iteration kernels (K8a + K8b), algorithmic bytes / CUDA-event time, PER GPU ------
    n_eval, n_upd = acc["n_pressure_eval"], acc["n_pressure_iter"]
    pa_ms = acc["predict_density_ms"] / max(n_eval, 1)
    pb_ms = acc["pressure_update_ms"] / max(n_upd, 1)
    it_bytes = nf_local * (BYTES["predict_density"] + BYTES["pressure_update"])  # this rank's particles vs ONE chip's peak
    it_ms = pa_ms + pb_ms
    achieved = it_bytes / (it_ms * 1e-3) / 1e9 if it_ms > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        traffic = (json.load(open(tp)).get(cfg) or {}).get("pair")
    roofline = {"bound": "hbm", "kernel": "predicted-density evaluation + pressure velocity update (one DFSPH pressure iteration), rank 0's GPU",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "bytes_per_launch": it_bytes, "particles_on_this_gpu": nf_local, "ms_per_launch_pair": it_ms,
                "predict_density_ms": pa_ms, "pressure_update_ms": pb_ms,
                "limiter": "L1TEX gather wavefronts + FP32 issue, not DRAM (see DESIGN.md)"}

    # ---- cpu_baseline: oracle port on a bounded sample of the same workload ----------------------------------------
    cpu = None
    if not args.no_cpu:
        edge = cpu_sample_edge(cfg, args.n, args.ref_n)
        csc = build_scene(cfg, edge, 1)
        cnf = sum(len(f["positions"]) for f in csc["fluids"])
        probe = build_scene(cfg, min(edge or 64, 64), 1) if cfg in ("c2", "c3", "c4") else csc
        cv, cms, threads, _ = run_oracle(csc, args.cpu_steps, 1, best_oracle_threads(probe))
        cpu = {"value": cv, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "%s generator at %d fluid particles (%s), 1+%d steps, %.0f ms/step" %
                         (cfg.upper(), cnf, "the whole workload" if cnf == nf else "bounded sample", args.cpu_steps, cms)}
        cpu.update(cpu_extras(cfg))
    phases = {k: acc[k] / args.steps for k in sorted(acc) if k.endswith("_ms")}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": args.steps, "warmup": warm,
            "ms_per_step": dev_s / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": static_config(cfg, args.n, world_size),
            "parallelism": "1 GPU" if world_size == 1 else
                           "%d x-slabs, 1-cell ghost columns exchanged per sub-iteration, %d exchanges/step" % (world_size, st["n_exchanges"]),
            "fluid_particles_per_gpu": nf // world_size,
            "iterations_per_step_mean": [float(np.mean([i[0] for i in iters])), float(np.mean([i[1] for i in iters]))],
            "phases": phases, "wall_ms_per_step": wall / args.steps * 1e3,
            "per_step_ms_rank0": {"step": [p[0] for p in per_step[:64]], "grid": [p[1] for p in per_step[:64]]},
            "grid_order": grid_order,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps, "api": "sph_fluid_write + sph_world_step + sph_fluid_read (pinned host buffers), all ranks"},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "parity": parity, "settled": settled, "single_gpu_slice": slice_ref}
    print(json.dumps(line), flush=True)
    if parity is not None and not parity.get("ok", False):
        sys.stderr.write("PARITY FAILED: %s\n" % json.dumps(parity))
        return 3
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default=None, choices=["c1", "c2", "c3", "c4", "c5"],
                    help="default: c3 on one GPU, c4 (4M particles per GPU) on several")
    ap.add_argument("--n", type=int, default=0, help="override lattice edge (testing)")
    ap.add_argument("--ref-n", type=int, default=0, help="lattice edge of the bounded CPU sample (0 = automatic)")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--parity-n", type=int, default=64, help="lattice edge of the in-line parity scene (64 -> 262144 particles)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-settled", action="store_true")
    ap.add_argument("--no-slice-ref", action="store_true", help="N > 1: skip the 1-GPU run of one rank's slice")
    ap.add_argument("--fast-sort", action="store_true", help="skip the deterministic in-cell ordering")
    ap.add_argument("--force-iters", type=int, nargs=2, default=None)
    ap.add_argument("--backend", type=int, default=0, help="0 = L1 gathers (default), 1 = tile/TMA shared-memory gathers")
    ap.add_argument("--grid-order", default="auto", choices=["auto", "h", "rows"],
                    help="particle order of the counting sort: h = cells of width h (z fastest), rows = x / y binned at h / 2 (SALVA_B200_XYSUB=2); "
                         "auto (one GPU, DFSPH dam-break configs) = run both as short parity-checked probes and keep the faster one")
    ap.add_argument("--probe", action="store_true", help="internal: short run of one grid order (no CPU arm, no e2e loop)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write each fluid's positions and velocities as DIR/fluid<k>_{positions,velocities}.npy "
                         "(f32, a fixed seeded sample above %d particles in all); one GPU, native arm only" % DUMP_MAX_PARTICLES)
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world_size = int(os.environ.get("WORLD_SIZE", 1))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or world_size > 1):
        ap.error("--dump-outputs needs the native arm on one GPU")
    if args.impl == "reference":
        reference_arm(args, rank, world_size)
        return 0
    try:
        rc = native_arm(args, rank, world_size)
    except BaseException:
        # one rank failing must not leave its peers (or its own tear-down) waiting in a collective: report and leave at once;
        # torchrun then stops the other ranks
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        sys.stdout.flush()
        os._exit(1)
    if world_size > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
        sys.stdout.flush()
        os._exit(rc)   # skip interpreter tear-down: destroying NCCL communicators of already-finished peers can block
    return rc


if __name__ == "__main__":
    sys.exit(main())
