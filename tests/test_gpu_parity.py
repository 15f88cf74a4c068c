"""GPU parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle on the
same seeded inputs (SURVEY.md §8c tolerances, written next to each assert).

  - neighbour counts: exact (integer)
  - rho, alpha, div, rho*: rel <= 1e-5 (+ abs 1e-6 * rho0 scale)
  - N-step trajectories with forced iteration counts: max|dx| <= 1e-3 h, max|dv| <= 1e-3 h/dt
"""
import numpy as np
import pytest

from oracle.oracle import OracleWorld
from salva_b200 import DFSPHSolver, IISPHSolver, LiquidWorld, scenes

pytestmark = pytest.mark.gpu


def _pair(scene, solver=0, **kw):
    r = scene["particle_radius"]
    gpu = LiquidWorld(DFSPHSolver() if solver == 0 else IISPHSolver(), particle_radius=r, smoothing_factor=2.0, **kw)
    cpu = OracleWorld(r, 2.0, solver=solver)
    fg, bg = scenes.populate(gpu, scene)
    fc, bc = scenes.populate(cpu, scene)
    return gpu, cpu, fg, fc, bg, bc


def _small_scene(seed=3, forces=(), two_fluids=False, nx=12, ny=10, nz=9, compress=0.93, vel_sigma=0.2, want_forces=False):
    r = 0.05
    rng = np.random.default_rng(seed)
    pts = scenes.jitter(scenes.block_lattice(nx, ny, nz, r * compress), r, seed, amplitude=0.3)
    vel = rng.normal(0, vel_sigma, pts.shape).astype(np.float32)
    tank = scenes.open_tank((-r, -r, -r), (nx * 2 * r + r, 1.0, nz * 2 * r + r), r)
    fluids = [dict(positions=pts, velocities=vel, density0=1000.0, forces=list(forces))]
    if two_fluids:
        up = scenes.jitter(scenes.block_lattice(nx, 4, nz, r * compress, origin=(0.0, ny * 2 * r * compress, 0.0)), r,
                           seed + 1, amplitude=0.3)
        fluids.append(dict(positions=up, velocities=rng.normal(0, vel_sigma, up.shape).astype(np.float32),
                           density0=800.0, forces=list(forces)))
    return dict(particle_radius=r, fluids=fluids, boundaries=[dict(positions=tank, want_forces=want_forces)])


def _rel(a, b, scale=None):
    scale = np.abs(b).max() if scale is None else scale
    return float(np.abs(a - b).max() / max(scale, 1e-30))


def test_single_pass_quantities_match_oracle():
    sc = _small_scene()
    gpu, cpu, fg, fc, bg, bc = _pair(sc)
    for w in (gpu, cpu):
        w.force_iterations(1, 1)
        w.step(0.005)
    f, o = fg[0], fc[0]
    assert np.array_equal(gpu.debug(f, "num_fluid_contacts"), cpu.debug(o, "num_fluid_contacts"))      # exact
    assert np.array_equal(gpu.debug(f, "num_boundary_contacts"), cpu.debug(o, "num_boundary_contacts"))  # exact
    assert _rel(gpu.debug(f, "density"), cpu.debug(o, "density")) <= 1e-5
    assert _rel(gpu.debug(f, "alpha"), cpu.debug(o, "alpha")) <= 1e-5
    # 1e-4, not the 1e-5 of rho / alpha / rho*: sum_j m (v_i - v_j) . grad W cancels to ~1 % of its terms, so the one-ulp
    # difference per term (g * x_ij here, dir * W' in the reference) is amplified ~100x relative to max|div| (DESIGN.md 4b)
    assert _rel(gpu.debug(f, "divergence"), cpu.debug(o, "divergence")) <= 1e-4
    assert _rel(gpu.debug(f, "predicted_density"), cpu.debug(o, "predicted_density")) <= 1e-5
    volg, _ = gpu.read_boundary(bg[0])
    volc, _ = cpu.read_boundary(bc[0])
    assert _rel(volg, volc) <= 1e-5
    sg, so = gpu.stats(), cpu.stats()
    assert sg["n_contacts"] == so["n_contacts"]


def test_list_capacity_regrows_behind_speculative_density_pass():
    """A crowded cell overflows the initial contact-list capacity: the neighbour phase must rebuild the lists (the density
    pass it had already enqueued speculatively is discarded and repeated) and still match the oracle."""
    r = 0.05
    h = 4 * r
    rng = np.random.default_rng(11)
    blob = (rng.random((400, 3)) * 0.9 * h + 0.05 * h).astype(np.float32)          # 400 particles in ONE cell
    rest = scenes.jitter(scenes.block_lattice(6, 6, 6, r, origin=(2.0, 0.0, 0.0)), r, 5, amplitude=0.2)
    pts = np.concatenate([blob, rest]).astype(np.float32)
    sc = dict(particle_radius=r, fluids=[dict(positions=pts, velocities=np.zeros_like(pts), density0=1000.0, forces=[])],
              boundaries=[])
    gpu, cpu, fg, fc, _, _ = _pair(sc)
    for w in (gpu, cpu):
        w.force_iterations(1, 1)
        w.step(1e-5)
    assert gpu.stats()["max_neighbors"] >= 400
    assert np.array_equal(gpu.debug(fg[0], "num_fluid_contacts"), cpu.debug(fc[0], "num_fluid_contacts"))
    assert _rel(gpu.debug(fg[0], "density"), cpu.debug(fc[0], "density")) <= 2e-5
    assert _rel(gpu.debug(fg[0], "alpha"), cpu.debug(fc[0], "alpha")) <= 1e-4
    assert _rel(gpu.debug(fg[0], "divergence"), cpu.debug(fc[0], "divergence")) <= 1e-3 or np.abs(cpu.debug(fc[0], "divergence")).max() == 0


@pytest.mark.parametrize("forces", [(), (scenes.xsph_viscosity(0.5, 0.3),), (scenes.artificial_viscosity(1.0, 0.5),),
                                    (scenes.akinci2013_surface_tension(1.0, 0.7),)],
                         ids=["none", "xsph", "artificial", "akinci2013"])
@pytest.mark.parametrize("backend", [0, 1], ids=["l1-gather", "tile-tma"])
def test_trajectory_forced_iterations(forces, backend):
    sc = _small_scene(seed=5, forces=forces)
    gpu, cpu, fg, fc, _, _ = _pair(sc, gather_backend=backend)
    dt = 0.005
    for w in (gpu, cpu):
        w.force_iterations(2, 3)
    for _ in range(10):
        gpu.step(dt)
        cpu.step(dt)
    pg, vg = gpu.read_fluid(fg[0])
    pc, vc = cpu.read_fluid(fc[0])
    h = float(gpu.h)
    assert _rel(gpu.debug(fg[0], "acceleration"), cpu.debug(fc[0], "acceleration")) <= 1e-3
    assert np.abs(pg - pc).max() <= 1e-3 * h          # SURVEY §8c
    assert np.abs(vg - vc).max() <= 1e-3 * h / dt


@pytest.mark.parametrize("two_fluids", [False, True], ids=["one-fluid", "two-fluids"])
@pytest.mark.parametrize("forces", [(scenes.he2014_surface_tension(40.0, 30.0),), (scenes.wcsph_surface_tension(2.0),)],
                         ids=["he2014", "wcsph"])
def test_surface_tension_rows_next(forces, two_fluids):
    """SURVEY §8(f).3: He2014SurfaceTension (he2014_surface_tension.rs) and the fluid term of WCSPHSurfaceTension
    (wcsph_surface_tension.rs:45-63), incl. the He2014 boundary reaction written through Boundary::apply_force."""
    sc = _small_scene(seed=23, forces=forces, two_fluids=two_fluids, want_forces=True)
    gpu, cpu, fg, fc, bg, bc = _pair(sc)
    dt = 0.004
    for w in (gpu, cpu):
        w.force_iterations(2, 3)
    for _ in range(6):
        gpu.step(dt)
        cpu.step(dt)
    h = float(gpu.h)
    for a, b in zip(fg, fc):
        ag, ac = gpu.debug(a, "acceleration"), cpu.debug(b, "acceleration")
        assert np.abs(ac - np.array([0, -9.81, 0], np.float32)).max() > 1.0      # the force is actually acting
        assert _rel(ag, ac) <= 1e-3
        pg, vg = gpu.read_fluid(a)
        pc, vc = cpu.read_fluid(b)
        assert np.abs(pg - pc).max() <= 1e-3 * h
        assert np.abs(vg - vc).max() <= 1e-3 * h / dt
    _, fgp = gpu.read_boundary(bg[0])
    _, fcp = cpu.read_boundary(bc[0])
    assert _rel(fgp, fcp) <= 1e-3


@pytest.mark.parametrize("two_fluids", [False, True], ids=["one-fluid", "two-fluids"])
@pytest.mark.parametrize("max_iter", [1, 3])
def test_dfsph_viscosity_row_a16(two_fluids, max_iter):
    """viscosity/dfsph_viscosity.rs: betas (6x6 LU inverse per particle), strain-rate targets, Jacobi loop.  Upstream's
    loop amplifies the strain-rate error ~60x per iteration on such scenes (tests/test_oracle_vs_numpy.py), so parity is
    checked relative to the size of the force after a bounded number of iterations."""
    sc = _small_scene(seed=31, forces=(scenes.dfsph_viscosity(0.5, 1, max_iter, 0.01),), two_fluids=two_fluids)
    gpu, cpu, fg, fc, _, _ = _pair(sc)
    for w in (gpu, cpu):
        w.force_iterations(2, 3)
    for _ in range(2):                                    # step 1 has dt = inv_dt = 0 in the force phase
        gpu.step(0.004)
        cpu.step(0.004)
    g = np.array([0.0, -9.81, 0.0], np.float32)
    for a, b in zip(fg, fc):
        ag, ac = gpu.debug(a, "acceleration"), cpu.debug(b, "acceleration")
        scale = np.abs(ac - g).max()
        assert scale > 100.0
        assert np.abs(ag - ac).max() <= 2e-3 * scale
        _, vg = gpu.read_fluid(a)
        _, vc = cpu.read_fluid(b)
        assert np.abs(vg - vc).max() <= 2e-3 * np.abs(vc).max()


def test_dfsph_viscosity_coefficient_range_is_checked():
    from salva_b200 import SphError
    gpu = LiquidWorld(particle_radius=0.05)
    f = gpu.add_fluid(np.zeros((4, 3), np.float32) + np.arange(4, dtype=np.float32)[:, None] * 0.1)
    with pytest.raises(SphError):                         # assert! dfsph_viscosity.rs:106-110
        gpu.push_force(f, *scenes.dfsph_viscosity(1.5))


def test_xsph_fusion_falls_back_when_the_loop_ends_with_an_update():
    """divergence_solve that runs out of iterations ends with an UPDATE (dfsph_solver.rs:474-502): the XSPH sums of its
    last evaluation are stale, so the separate XSPH pass must run."""
    sc = _small_scene(seed=41, forces=(scenes.xsph_viscosity(0.5, 0.0),))
    solver = DFSPHSolver()
    solver.max_divergence_iter, solver.max_divergence_error = 2, 1e-9      # never converges: exactly 2 updates
    gpu = LiquidWorld(solver, particle_radius=sc["particle_radius"], smoothing_factor=2.0)
    cpu = OracleWorld(sc["particle_radius"], 2.0, max_divergence_iter=2, max_divergence_error=1e-9)
    fg, _ = scenes.populate(gpu, sc)
    fc, _ = scenes.populate(cpu, sc)
    dt = 0.005
    for _ in range(6):
        gpu.step(dt)
        cpu.step(dt)
    assert gpu.stats()["n_divergence_iter"] == 2 and gpu.stats()["n_divergence_eval"] == 2
    pg, vg = gpu.read_fluid(fg[0])
    pc, vc = cpu.read_fluid(fc[0])
    h = float(gpu.h)
    assert _rel(gpu.debug(fg[0], "acceleration"), cpu.debug(fc[0], "acceleration")) <= 1e-3
    assert np.abs(pg - pc).max() <= 1e-3 * h
    assert np.abs(vg - vc).max() <= 1e-3 * h / dt


@pytest.mark.parametrize("mode", ["forced", "free", "boundary-term-fallback"])
def test_xsph_fused_with_divergence_evaluation(mode):
    """The XSPH sums ride with the divergence loop's stand-alone evaluations
    (k_vel_divergence_xsph_u) and k_fold_velocities applies the last ones; with a boundary coefficient the engine must
    fall back to the separate pass.  Same tolerances as the plain trajectory test."""
    forces = (scenes.xsph_viscosity(0.5, 0.3 if mode == "boundary-term-fallback" else 0.0),)
    sc = _small_scene(seed=37, forces=forces)
    gpu, cpu, fg, fc, _, _ = _pair(sc)
    dt = 0.005
    if mode != "free":
        for w in (gpu, cpu):
            w.force_iterations(2, 3)
    for _ in range(8):
        gpu.step(dt)
        cpu.step(dt)
    pg, vg = gpu.read_fluid(fg[0])
    pc, vc = cpu.read_fluid(fc[0])
    h = float(gpu.h)
    ac = cpu.debug(fc[0], "acceleration")
    assert np.abs(ac - np.array([0, -9.81, 0], np.float32)).max() > 0.5     # XSPH is acting
    assert _rel(gpu.debug(fg[0], "acceleration"), ac) <= 1e-3
    assert np.abs(pg - pc).max() <= 1e-3 * h
    assert np.abs(vg - vc).max() <= 1e-3 * h / dt


def test_wcsph_boundary_coefficient_is_rejected():
    from salva_b200 import SphError
    gpu = LiquidWorld(particle_radius=0.05)
    f = gpu.add_fluid(np.zeros((4, 3), np.float32) + np.arange(4, dtype=np.float32)[:, None] * 0.1)
    with pytest.raises(SphError):
        gpu.push_force(f, *scenes.wcsph_surface_tension(1.0, 0.5))


def test_particles_intersecting_aabb_matches_oracle():
    """liquid_world.rs:211-243: cells of the LAST step's grid, current positions, distance < particle_radius."""
    from salva_b200 import SphError
    sc = _small_scene(seed=29, vel_sigma=0.6)
    gpu, cpu, fg, fc, bg, bc = _pair(sc)
    boxes = [((0.13, -0.2, 0.11), (0.47, 0.33, 0.38)), ((-5.0, -5.0, -5.0), (5.0, 5.0, 5.0)), ((0.31, 0.2, 0.3), (0.32, 0.21, 0.31)),
             ((7.0, 7.0, 7.0), (8.0, 8.0, 8.0))]
    k, _, _ = gpu.particles_intersecting_aabb(*boxes[0])
    assert len(k) == 0                                   # before the first step the reference's grid is empty
    for w in (gpu, cpu):
        w.force_iterations(1, 2)
    for step in range(3):
        gpu.step(0.004)
        cpu.step(0.004)
        for mins, maxs in boxes:
            g = gpu.particles_intersecting_aabb(mins, maxs)
            c = cpu.particles_intersecting_aabb(mins, maxs)
            assert all(np.array_equal(a, b) for a, b in zip(g, c)), (step, mins)
    assert len(gpu.particles_intersecting_aabb(*boxes[1])[0]) > 1000
    # a host edit of positions keeps the stale cells but tests the new positions, exactly like the reference
    p, v = cpu.read_fluid(fc[0])
    p2 = (p + np.float32(0.03)).astype(np.float32)
    gpu.write_fluid(fg[0], p2, v)
    cpu.write_fluid(fc[0], p2, v)
    for mins, maxs in boxes[:3]:
        g = gpu.particles_intersecting_aabb(mins, maxs)
        c = cpu.particles_intersecting_aabb(mins, maxs)
        assert all(np.array_equal(a, b) for a, b in zip(g, c))
    gpu.append_particles(fg[0], np.array([[0.2, 0.5, 0.2]], np.float32))
    with pytest.raises(SphError):                        # structural edit pending: the old grid no longer applies
        gpu.particles_intersecting_aabb(*boxes[0])


@pytest.mark.parametrize("backend", [0, 1], ids=["l1-gather", "tile-tma"])
def test_two_fluids_with_groups_and_free_running_iterations(backend):
    sc = _small_scene(seed=9, forces=(scenes.xsph_viscosity(0.5, 0.0),), two_fluids=True)
    gpu, cpu, fg, fc, _, _ = _pair(sc, gather_backend=backend)
    for _ in range(4):
        gpu.step(0.005)
        cpu.step(0.005)
        sg, so = gpu.stats(), cpu.stats()
        assert sg["n_divergence_iter"] == so["n_divergence_iter"]
        assert sg["n_pressure_iter"] == so["n_pressure_iter"]
        assert sg["last_density_error"] == pytest.approx(so["last_density_error"], rel=1e-3, abs=1e-7)
    h = float(gpu.h)
    for a, b in zip(fg, fc):
        pg, vg = gpu.read_fluid(a)
        pc, vc = cpu.read_fluid(b)
        assert np.array_equal(gpu.debug(a, "num_fluid_contacts"), cpu.debug(b, "num_fluid_contacts"))
        assert np.abs(pg - pc).max() <= 1e-3 * h


def test_interaction_groups_filter_pairs():
    """Two fluids whose groups do not match never see each other (contacts.rs:355-362)."""
    sc = _small_scene(seed=11, two_fluids=True)
    sc["fluids"][0].update(memberships=1, filter=1)
    sc["fluids"][1].update(memberships=2, filter=2)
    sc["boundaries"][0].update(memberships=3, filter=3)
    gpu, cpu, fg, fc, _, _ = _pair(sc)
    for w in (gpu, cpu):
        w.force_iterations(1, 2)
        w.step(0.005)
    for a, b in zip(fg, fc):
        assert np.array_equal(gpu.debug(a, "num_fluid_contacts"), cpu.debug(b, "num_fluid_contacts"))
        assert _rel(gpu.debug(a, "density"), cpu.debug(b, "density")) <= 1e-5


@pytest.mark.parametrize("two_fluids", [False, True], ids=["one-fluid", "two-fluids"])
def test_iisph_forced_iterations_trajectory(two_fluids):
    """IISPHSolver::step iisph_solver.rs:643-711 (row a23): dii, aii, relaxed Jacobi on pressures, warm start."""
    # NOTE: ArtificialViscosity's boundary reaction uses the RUNNING boundary_acc (artificial_viscosity.rs:117), which
    # depends on the (unspecified) contact order, so boundary forces are compared with XSPH's boundary term instead.
    sc = _small_scene(seed=23, forces=(scenes.artificial_viscosity(1.0, 0.0), scenes.xsph_viscosity(0.3, 0.4)),
                      two_fluids=two_fluids, want_forces=True)
    gpu, cpu, fg, fc, bg, bc = _pair(sc, solver=1)
    dt = 0.005
    for w in (gpu, cpu):
        w.force_iterations(-1, 4)
    for _ in range(6):
        gpu.step(dt)
        cpu.step(dt)
    h = float(gpu.h)
    for a, b in zip(fg, fc):
        pg, vg = gpu.read_fluid(a)
        pc, vc = cpu.read_fluid(b)
        assert _rel(gpu.debug(a, "pressure"), cpu.debug(b, "pressure")) <= 2e-3
        assert _rel(gpu.debug(a, "predicted_density"), cpu.debug(b, "predicted_density")) <= 1e-5
        assert np.abs(pg - pc).max() <= 1e-3 * h
        assert np.abs(vg - vc).max() <= 1e-3 * h / dt
    _, fgp = gpu.read_boundary(bg[0])
    _, fcp = cpu.read_boundary(bc[0])
    assert _rel(fgp, fcp) <= 2e-3


def test_iisph_free_running_iteration_counts():
    sc = _small_scene(seed=29)
    gpu, cpu, fg, fc, _, _ = _pair(sc, solver=1)
    for _ in range(5):
        gpu.step(0.005)
        cpu.step(0.005)
        assert gpu.stats()["n_pressure_iter"] == cpu.stats()["n_pressure_iter"]
    pg, _ = gpu.read_fluid(fg[0])
    pc, _ = cpu.read_fluid(fc[0])
    assert np.abs(pg - pc).max() <= 1e-3 * float(gpu.h)


@pytest.mark.parametrize("nonlinear", [True, False], ids=["nonlinear", "linear"])
def test_becker2009_elasticity_trajectory(nonlinear):
    """Becker2009Elasticity::solve becker2009_elasticity.rs:84-334 (row a15): rest lists keyed by original index,
    rotation extraction (nalgebra from_matrix_eps restated), corotated stress, pairwise forces."""
    sc = _small_scene(seed=31, forces=(scenes.becker2009_elasticity(1.0e5, 0.3, nonlinear),), nx=8, ny=8, nz=8, compress=1.0, vel_sigma=0.05)
    gpu, cpu, fg, fc, _, _ = _pair(sc)
    dt = 0.002
    for w in (gpu, cpu):
        w.force_iterations(1, 2)
    for _ in range(8):
        gpu.step(dt)
        cpu.step(dt)
    pg, vg = gpu.read_fluid(fg[0])
    pc, vc = cpu.read_fluid(fc[0])
    h = float(gpu.h)
    acc_c = cpu.debug(fc[0], "acceleration")
    assert np.abs(acc_c - np.array([0, -9.81, 0], np.float32)).max() > 1.0  # elasticity is doing something
    assert _rel(gpu.debug(fg[0], "acceleration"), acc_c) <= 2e-3
    assert np.abs(pg - pc).max() <= 1e-3 * h
    assert np.abs(vg - vc).max() <= 1e-3 * h / dt


def test_config_c5_small_iisph_two_fluids_elastic():
    """BASELINE.json configs[4] at reduced size: IISPH + ArtificialViscosity + Becker2009 on two stacked fluids."""
    sc = scenes.scene_c5(8)
    gpu, cpu, fg, fc, _, _ = _pair(sc, solver=1)
    for w in (gpu, cpu):
        w.force_iterations(-1, 3)
    for _ in range(5):
        gpu.step(sc["dt"])
        cpu.step(sc["dt"])
    h = float(gpu.h)
    for a, b in zip(fg, fc):
        pg, vg = gpu.read_fluid(a)
        pc, vc = cpu.read_fluid(b)
        assert np.abs(pg - pc).max() <= 1e-3 * h
        assert np.abs(vg - vc).max() <= 1e-3 * h / sc["dt"]


def test_config_c1_basic3_ten_steps():
    """BASELINE.json configs[0]: examples3d/basic3.rs scene, reference CPU (f32)."""
    sc = scenes.scene_c1()
    gpu, cpu, fg, fc, _, _ = _pair(sc)
    for w in (gpu, cpu):
        w.force_iterations(1, 2)
    for _ in range(10):
        gpu.step(sc["dt"])
        cpu.step(sc["dt"])
    pg, vg = gpu.read_fluid(fg[0])
    pc, vc = cpu.read_fluid(fc[0])
    h = float(gpu.h)
    assert np.array_equal(gpu.debug(fg[0], "num_fluid_contacts"), cpu.debug(fc[0], "num_fluid_contacts"))
    assert np.abs(pg - pc).max() <= 1e-3 * h
    assert np.abs(vg - vc).max() <= 1e-3 * h / sc["dt"]


def test_host_edits_append_delete_roundtrip():
    """fluids_mut() edits, Fluid::add_particles (fluid.rs:126-150) and deletion (fluid.rs:71-98) keep ORIGINAL
    index order and match the oracle's host-side semantics."""
    sc = _small_scene(seed=13, nx=8, ny=6, nz=6)
    gpu, cpu, fg, fc, _, _ = _pair(sc)
    f, o = fg[0], fc[0]
    rng = np.random.default_rng(1)
    for w in (gpu, cpu):
        w.force_iterations(1, 2)
        w.step(0.005)
    p0, v0 = gpu.read_fluid(f)
    newv = (v0 * 0.5).astype(np.float32)
    extra = (p0[:20] + np.array([0.0, 0.8, 0.0], np.float32)).astype(np.float32)
    mask = np.zeros(len(p0), np.uint8)
    mask[rng.choice(len(p0), 30, replace=False)] = 1
    for w, h in ((gpu, f), (cpu, o)):
        w.write_fluid(h, velocities=newv)
        w.delete_particles(h, mask)
        w.append_particles(h, extra)
        w.step(0.005)
        w.step(0.005)
    assert gpu.num_particles(f) == cpu.num_particles(o) == len(p0) - 30 + 20
    pg, vg = gpu.read_fluid(f)
    pc, vc = cpu.read_fluid(o)
    assert np.abs(pg - pc).max() <= 1e-3 * float(gpu.h)


@pytest.mark.parametrize("backend", [0, 1], ids=["l1-gather", "tile-tma"])
def test_boundary_forces_accumulate_like_reference(backend):
    """Boundary::apply_force (boundary.rs:62-67) writers: dfsph_solver.rs:269-272,403-405 and the force plugins."""
    sc = _small_scene(seed=17, forces=(scenes.xsph_viscosity(0.5, 0.3),), want_forces=True)
    gpu, cpu, fg, fc, bg, bc = _pair(sc, gather_backend=backend)
    for w in (gpu, cpu):
        w.force_iterations(2, 3)
    for _ in range(3):
        gpu.step(0.005)
        cpu.step(0.005)
    _, fgp = gpu.read_boundary(bg[0])
    _, fcp = cpu.read_boundary(bc[0])
    assert np.abs(fcp).max() > 0
    assert _rel(fgp, fcp) <= 1e-3


def test_boundary_rewrite_between_steps():
    """CouplingManager::update_boundaries rewrites boundary particles every substep (coupling_manager.rs:12-20);
    the engine caches the boundary sort / volumes only while they are unchanged."""
    sc = _small_scene(seed=19, forces=(scenes.xsph_viscosity(0.5, 0.3),))
    gpu, cpu, fg, fc, bg, bc = _pair(sc)
    tank = sc["boundaries"][0]["positions"]
    for w in (gpu, cpu):
        w.force_iterations(1, 2)
    for k in range(6):
        if k in (2, 3, 5):
            shift = np.array([0.004 * k, 0.002 * k, -0.003 * k], np.float32)
            vel = np.tile(np.array([0.8, 0.4, -0.6], np.float32), (len(tank), 1))
            for w, b in ((gpu, bg[0]), (cpu, bc[0])):
                w.write_boundary(b, positions=(tank + shift).astype(np.float32), velocities=vel)
        gpu.step(0.005)
        cpu.step(0.005)
    pg, vg = gpu.read_fluid(fg[0])
    pc, vc = cpu.read_fluid(fc[0])
    volg, _ = gpu.read_boundary(bg[0])
    volc, _ = cpu.read_boundary(bc[0])
    assert _rel(volg, volc) <= 1e-5
    assert np.array_equal(gpu.debug(fg[0], "num_boundary_contacts"), cpu.debug(fc[0], "num_boundary_contacts"))
    assert np.abs(pg - pc).max() <= 1e-3 * float(gpu.h)
    assert gpu.stats()["n_contacts"] == cpu.stats()["n_contacts"]


def test_user_defined_host_force_plugin():
    """NonPressureForce trait objects with arbitrary host code (nonpressure_force.rs:10-30): the custom force field of
    examples3d/custom_forces3.rs:66-90 (acc += dir / dist towards an origin), pushed BETWEEN two built-in forces."""
    origin = np.array([0.3, 0.6, 0.2], np.float32)

    def solve(dt, inv_dt, h, pos, vel, dens, acc):
        d = origin - pos
        sq = (d * d).sum(axis=1)
        ok = sq > 0.1 * 0.1
        dist = np.sqrt(sq[ok])
        acc[ok] += (d[ok] / dist[:, None]) / dist[:, None]

    sc = _small_scene(seed=37)
    gpu, cpu, fg, fc, _, _ = _pair(sc)
    for w, f in ((gpu, fg[0]), (cpu, fc[0])):
        w.push_force(f, *scenes.xsph_viscosity(0.5, 0.0))
        w.push_host_force(f, solve)
        w.push_force(f, *scenes.artificial_viscosity(1.0, 0.0))
        w.force_iterations(1, 2)
    for _ in range(4):
        gpu.step(0.005)
        cpu.step(0.005)
    pg, vg = gpu.read_fluid(fg[0])
    pc, vc = cpu.read_fluid(fc[0])
    assert _rel(gpu.debug(fg[0], "acceleration"), cpu.debug(fc[0], "acceleration")) <= 1e-3
    assert np.abs(pg - pc).max() <= 1e-3 * float(gpu.h)


def test_deterministic_mode_is_bit_reproducible():
    sc = _small_scene(seed=21)
    outs = []
    for _ in range(2):
        gpu = LiquidWorld(particle_radius=sc["particle_radius"], deterministic=True)
        fg, _ = scenes.populate(gpu, sc)
        for _ in range(5):
            gpu.step(0.005)
        outs.append(gpu.read_fluid(fg[0]))
        gpu.close()
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])


def test_error_paths():
    from salva_b200 import SphError
    gpu = LiquidWorld(particle_radius=0.05)
    f = gpu.add_fluid(np.array([[0, 0, 0], [np.nan, 0, 0]], np.float32))
    with pytest.raises(SphError) as e:
        gpu.step(0.005)
    assert e.value.status == 1
    with pytest.raises(SphError):
        gpu.read_fluid(f + 7)


def test_parity_at_110k_particles_through_the_bench_block():
    """The same GPU-vs-oracle block every bench line carries (bench.py parity_vs_oracle), at 48^3 = 110 592 particles of the
    C3 generator: contact counts exact on identical inputs, 3-step trajectory within the SURVEY 8(c) tolerances."""
    import bench
    res = bench.parity_vs_oracle("c3", 0, edge=48, steps=3)
    assert res["n"] == 48 ** 3 and res["contacts_equal"] is True
    assert res["max_dx_over_h"] <= 1e-3 and res["max_rel_rho"] <= 1e-5 and res["max_dv_over_h_dt"] <= 1e-3
    assert res["ok"]
