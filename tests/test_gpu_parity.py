"""GPU parity: the CUDA engine (through the Python surface -> C ABI) against the CPU oracle.

Tolerances (fp32 path; the reference itself runs Taichi fast_math and unordered atomics, so
bitwise parity with it is not defined -- SURVEY Q7/Q10):
  * integer work (cell ids, prefix sums, sort permutation): bit-exact;
  * per-kernel sums from an identical sorted state: 2e-5 of the field's max magnitude
    (the engine multiplies by 1/h and uses multiply chains where the oracle divides / calls powf);
  * trajectories: max |dx| / particle diameter after N steps below 1e-3 and within 20x of the
    oracle's own fp32-vs-fp64 drift over the same N steps.
"""
import numpy as np
import pytest

from tests.helpers import jitter, mixed_scene, order_by_x0

pytestmark = pytest.mark.gpu

REL = 2e-5


def _pair(scene_dict, seed=None, amp=0.004, register_blocks=()):
    from oracle.sph_oracle import OracleSim
    from sph_taichi_b200 import ParticleSystem, SimConfig

    o = OracleSim(scene_dict)
    cfg = SimConfig(scene_dict)
    ps = ParticleSystem(cfg)
    for oid in register_blocks:  # treat a RigidBlock as a shape-matched body in both
        o.object_id_rigid_body.add(oid)
        ps.object_id_rigid_body.add(oid)
    o.dyn_ids = sorted(i for i in o.object_id_rigid_body if o.object_collection[i]["isDynamic"])
    if seed is not None:
        jitter(o, amp, seed=seed)
        ps.x.from_numpy(o.x)
        ps.v.from_numpy(o.v)
    solver = ps.build_solver()
    return o, ps, solver


def _maxrel(a, b):
    scale = max(float(np.abs(b).max()), 1e-30)
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max()) / scale


def test_neighbor_build_bit_exact():
    o, ps, _ = _pair(mixed_scene(), seed=5)
    o.initialize_particle_system()
    ps.initialize_particle_system()
    assert np.array_equal(ps.grid_ids.to_numpy(), o.grid_ids)
    assert np.array_equal(ps.grid_particles_num.to_numpy(), o.grid_particles_num)
    for k in ("x", "x_0", "v", "object_id", "material", "is_dynamic", "color", "m", "m_V", "density"):
        assert np.array_equal(getattr(ps, k).to_numpy(), getattr(o, k)), k
    # idempotent: re-sorting a sorted state changes nothing
    before = ps.x.to_numpy().copy()
    ps.initialize_particle_system()
    assert np.array_equal(ps.x.to_numpy(), before)


@pytest.mark.parametrize("dims,n", [((8, 8, 8), 1), ((61, 7, 43), 5000), ((200, 100, 150), 200000)])
def test_prefix_sum_against_numpy(dims, n):
    """Decoupled look-back scan == np.cumsum for ragged / multi-tile / sparse grids."""
    from sph_taichi_b200 import ParticleSystem, SimConfig, scene

    h = 0.04
    dom = [d * h for d in dims]
    sc = scene.dam_break_box([1, 1, 1], domain_end=dom, start=[0.05, 0.05, 0.05])
    ps = ParticleSystem(SimConfig(sc))
    assert ps.particle_max_num == 1
    # the public surface has no emitter, so exercise big inputs through a fresh block scene
    rng = np.random.default_rng(n)
    cnt = max(1, int(round(n ** (1 / 3))))
    sc2 = scene.dam_break_box([cnt, cnt, cnt], domain_end=dom, start=[0.05, 0.05, 0.05], radius=0.01)
    ps2 = ParticleSystem(SimConfig(sc2))
    m = ps2.particle_max_num
    x = (rng.uniform(0.0, 1.0, size=(m, 3)) * (np.array(dom) - 1e-3)).astype(np.float32)
    x[: m // 4] = x[0]  # heavy collisions in one cell
    ps2.x.from_numpy(x)
    ps2.initialize_particle_system()
    cells = (x / np.float32(h)).astype(np.int32)
    g = [int(v) for v in ps2.grid_num]  # ceil(dom / h) may exceed dims by one through rounding
    flat = (cells[:, 0] * g[1] + cells[:, 1]) * g[2] + cells[:, 2]
    want = np.cumsum(np.bincount(flat, minlength=int(np.prod(g)))).astype(np.int32)
    assert np.array_equal(ps2.grid_particles_num.to_numpy(), want)
    assert np.array_equal(ps2.grid_ids.to_numpy(), np.sort(flat))
    perm = np.argsort(flat, kind="stable")
    assert np.array_equal(ps2.x.to_numpy(), x[perm])


def test_per_kernel_parity_mixed_scene():
    o, ps, solver = _pair(mixed_scene(), seed=1)
    o.initialize()
    solver.initialize()
    solid = o.material == 0
    assert np.array_equal(ps.x.to_numpy(), o.x)
    assert _maxrel(ps.m_V.to_numpy()[solid], o.m_V[solid]) < REL
    o.compute_densities(); solver.compute_densities()
    assert _maxrel(ps.density.to_numpy(), o.density) < REL
    o.compute_non_pressure_forces(); solver.compute_non_pressure_forces()
    assert _maxrel(ps.acceleration.to_numpy(), o.acceleration) < REL
    o.compute_pressure_forces(); solver.compute_pressure_forces()
    assert _maxrel(ps.pressure.to_numpy(), o.pressure) < 5 * REL  # x^7 amplifies the density ulps
    assert np.abs(o.acceleration).max() > 100.0
    assert _maxrel(ps.acceleration.to_numpy(), o.acceleration) < 5 * REL
    dyn_rigid = (o.material == 0) & (o.is_dynamic == 1)
    assert np.abs(o.acceleration[dyn_rigid] - np.array([0, -9.81, 0], np.float32)).max() > 1.0  # reactions present
    o.advect(); solver.advect()
    assert _maxrel(ps.x.to_numpy(), o.x) < 1e-6
    o.enforce_boundary_3D(1); solver.enforce_boundary_3D(1)
    o.enforce_boundary_3D(0); solver.enforce_boundary_3D(0)
    assert _maxrel(ps.x.to_numpy(), o.x) < 1e-6
    assert _maxrel(ps.v.to_numpy(), o.v) < 1e-4


def test_wall_clamp_and_reflection():
    from sph_taichi_b200 import scene
    o, ps, solver = _pair(scene.dam_break_box([6, 6, 6], domain_end=[0.4, 0.4, 0.4], start=[0.05, 0.05, 0.05]))
    rng = np.random.default_rng(2)
    x = o.x.copy()
    x[:50] = rng.uniform(-0.02, 0.05, size=(50, 3)).astype(np.float32) + np.float32(0.0)
    x[50:100, 1] = np.float32(0.4 - 0.04) + rng.uniform(-1e-3, 0.03, size=50).astype(np.float32)
    x[100] = [0.04, 0.36, 0.2]  # exactly on both thresholds
    o.x[:] = x
    o.v[:] = rng.uniform(-2, 2, size=o.v.shape).astype(np.float32)
    ps.x.from_numpy(o.x); ps.v.from_numpy(o.v)
    o.enforce_boundary_3D(1); solver.enforce_boundary_3D(1)
    assert np.array_equal(ps.x.to_numpy(), o.x)
    assert _maxrel(ps.v.to_numpy(), o.v) < 1e-6


def test_trajectory_cube8k_vs_oracle():
    from oracle.sph_oracle import OracleSim
    from sph_taichi_b200 import scene
    sc = scene.cube_8k()
    o, ps, solver = _pair(sc)
    o64 = OracleSim(sc, f64=True)
    steps = 60
    o.initialize(); o64.initialize(); solver.initialize()
    for _ in range(steps):
        o.step(); o64.step()
    solver.step(steps)
    d = 0.02
    ko, k64 = order_by_x0(o.x_0), order_by_x0(o64.x_0)
    floor = np.abs(o.x[ko] - o64.x[k64]).max() / d
    x, x0 = ps.x.to_numpy(), ps.x_0.to_numpy()
    kg = order_by_x0(x0)
    assert np.array_equal(x0[kg], o.x_0[ko])
    err = np.abs(x[kg] - o.x[ko]).max() / d
    err64 = np.abs(x[kg] - o64.x[k64]).max() / d
    assert err < 1e-3, (err, floor)
    assert err64 < max(20 * floor, 1e-4), (err64, floor)
    assert _maxrel(ps.v.to_numpy()[kg], o.v[ko]) < 1e-2


def test_fused_step_equals_method_sequence():
    from sph_taichi_b200.WCSPH import WCSPHSolver

    class Unfused(WCSPHSolver):
        def substep(self):  # overriding forces the reference's generic step() sequence
            super().substep()

    _, ps_a, sa = _pair(mixed_scene(), seed=9, register_blocks=(2,))
    _, ps_b, _ = _pair(mixed_scene(), seed=9, register_blocks=(2,))
    sb = Unfused(ps_b)
    sa.initialize(); sb.initialize()
    for _ in range(5):
        sa.step(); sb.step()
    for k in ("x", "v", "density", "pressure"):
        assert _maxrel(getattr(ps_a, k).to_numpy(), getattr(ps_b, k).to_numpy()) < 1e-5, k


def test_step_with_rigid_coupling_vs_oracle():
    """Static + dynamic rigid blocks; block 2 registered for shape matching in both."""
    o, ps, solver = _pair(mixed_scene(), seed=4, amp=0.002, register_blocks=(2,))
    o.initialize(); solver.initialize()
    assert _maxrel(ps.rigid_rest_cm[2], o.rest_cm[2]) < 1e-6
    steps = 25
    for _ in range(steps):
        o.step()
    solver.step(steps)
    ko = order_by_x0(o.x_0)
    x0 = ps.x_0.to_numpy()
    kg = order_by_x0(x0)
    assert np.array_equal(x0[kg], o.x_0[ko])
    assert np.array_equal(ps.object_id.to_numpy()[kg], o.object_id[ko])
    err = np.abs(ps.x.to_numpy()[kg] - o.x[ko]).max() / 0.02
    assert err < 2e-3, err
    rigid = (o.object_id[ko] == 2)
    assert np.abs(ps.x.to_numpy()[kg][rigid] - o.x[ko][rigid]).max() / 0.02 < 2e-3
    assert ps._engine.check_status() == 0


def test_rigid_solve_recovers_rotation_gpu():
    o, ps, solver = _pair(mixed_scene(with_static=False), register_blocks=(2,))
    solver.initialize()
    oid = 2
    x = ps.x.to_numpy(); x0 = ps.x_0.to_numpy(); sel = ps.object_id.to_numpy() == oid
    cm0 = ps.rigid_rest_cm[oid].astype(np.float64)
    th = 0.4
    Ry = np.array([[np.cos(th), 0, np.sin(th)], [0, 1, 0], [-np.sin(th), 0, np.cos(th)]])
    shift = np.array([0.01, 0.02, -0.005])
    x[sel] = ((x0[sel] - cm0) @ Ry.T + cm0 + shift).astype(np.float32)
    ps.x.from_numpy(x)
    ps.initialize_particle_system()
    R = solver.solve_constraints(oid).cpu().numpy()
    assert np.allclose(R, Ry, atol=1e-4)
    x1 = ps.x.to_numpy(); x01 = ps.x_0.to_numpy(); sel1 = ps.object_id.to_numpy() == oid
    assert np.allclose(x1[sel1], (x01[sel1] - cm0) @ Ry.T + cm0 + shift, atol=2e-5)


def test_rigid_solve_of_an_inverted_body_is_a_proper_rotation():
    """A mirrored (inverted) body: det A < 0.  ti.polar_decompose returns a PROPER rotation (its SVD keeps U and V
    rotations, the sign goes to the smallest singular value); the orthogonal polar factor would be a reflection."""
    o, ps, solver = _pair(mixed_scene(with_static=False), register_blocks=(2,))
    solver.initialize(); o.initialize()
    oid = 2
    x = ps.x.to_numpy(); x0 = ps.x_0.to_numpy(); sel = ps.object_id.to_numpy() == oid
    cm0 = ps.rigid_rest_cm[oid].astype(np.float64)
    th = 0.3
    Rz = np.array([[np.cos(th), -np.sin(th), 0], [np.sin(th), np.cos(th), 0], [0, 0, 1]])
    M = Rz @ np.diag([1.0, 0.8, -0.6])  # mirrored and squashed along z: det < 0, distinct singular values
    x[sel] = ((x0[sel] - cm0) @ M.T + cm0).astype(np.float32)
    ps.x.from_numpy(x)
    osel = o.object_id == oid
    o.x[osel] = ((o.x_0[osel] - cm0) @ M.T + cm0).astype(np.float32)
    ps.initialize_particle_system(); o.initialize_particle_system()
    R = solver.solve_constraints(oid).cpu().numpy().astype(np.float64)
    Ro = o.solve_constraints(oid).astype(np.float64)
    q = (x0[sel] - cm0).astype(np.float64)
    A = M @ (q.T @ q)  # sph_base.py:204-211 with equal masses: A = sum (x - c)(x_0 - c_0)^T = M sum q q^T
    U, s_, Vt = np.linalg.svd(A)
    want = U @ np.diag([1, 1, np.linalg.det(U @ Vt)]) @ Vt  # the sign goes to the SMALLEST singular value of A
    assert abs(np.linalg.det(R) - 1.0) < 1e-4 and np.allclose(R @ R.T, np.eye(3), atol=1e-4)
    assert np.allclose(R, want, atol=2e-3) and np.allclose(Ro, want, atol=2e-3)
    assert np.allclose(R, Ro, atol=1e-4)
    assert ps._engine.read_status() & 2 == 0


def test_dump_and_invariants_dragon_bath_full_size():
    """BASELINE cfg 2 at full size: size-independent properties after real steps."""
    from sph_taichi_b200 import ParticleSystem, SimConfig, scene
    ps = ParticleSystem(SimConfig(scene.dragon_bath()))
    assert ps.fluid_particle_num == 423500 and ps.particle_max_num == 423500 + ps.solid_particle_num
    solver = ps.build_solver()
    solver.initialize()
    solver.step(40)
    assert ps._engine.check_status() == 0
    gid = ps.grid_ids.to_numpy()
    assert np.all(np.diff(gid) >= 0)                       # sortedness
    gpn = ps.grid_particles_num.to_numpy()
    assert gpn[-1] == ps.particle_max_num                   # checksum of the scan
    assert np.array_equal(gpn, np.cumsum(np.bincount(gid, minlength=gpn.size)))
    d = ps.dump(0)
    assert d["position"].shape == (423500, 3)
    pad = np.float32(0.04)
    hi = (np.array([5.0, 3.0, 2.0]) - 0.04).astype(np.float32)
    assert (d["position"] >= pad).all() and (d["position"] <= hi).all()
    assert np.isfinite(d["velocity"]).all()
    # static dragon untouched, in its original order
    assert np.array_equal(np.sort(ps.dump(1)["position"], axis=0),
                          np.sort(ps.object_collection[1]["voxelizedPoints"].astype(np.float32), axis=0))
    rho = ps.density.to_numpy()[ps.material.to_numpy() == 1]
    assert rho.min() >= 1000.0 and rho.max() < 1300.0


def test_dragon_bath_full_size_against_oracle():
    """BASELINE cfg 2 at FULL size (441 996 particles), field by field against the oracle, particles matched
    by their immutable key (object id, x_0).  The engine first runs 320 steps (the column falls 0.06 m and hits
    the floor: clamps, pressure and viscosity are all active); that state is handed to the oracle and both
    advance 8 more steps."""
    from oracle.sph_oracle import OracleSim
    from sph_taichi_b200 import ParticleSystem, SimConfig, scene
    sc = scene.dragon_bath()
    ps = ParticleSystem(SimConfig(sc))
    solver = ps.build_solver()
    solver.initialize()
    o = OracleSim(sc)
    o.initialize()

    def keys(x0, oid):
        return np.lexsort((x0[:, 2], x0[:, 1], x0[:, 0], oid))

    solver.step(320)
    x0, oid = ps.x_0.to_numpy(), ps.object_id.to_numpy()
    kg, ko = keys(x0, oid), keys(o.x_0, o.object_id)
    assert np.array_equal(x0[kg], o.x_0[ko]) and np.array_equal(oid[kg], o.object_id[ko])
    o.x[ko] = ps.x.to_numpy()[kg]
    o.v[ko] = ps.v.to_numpy()[kg]
    steps = 8
    solver.step(steps)
    for _ in range(steps):
        o.step()
    assert ps._engine.check_status() == 0
    x, x0, oid = ps.x.to_numpy(), ps.x_0.to_numpy(), ps.object_id.to_numpy()
    kg, ko = keys(x0, oid), keys(o.x_0, o.object_id)
    assert np.array_equal(x0[kg], o.x_0[ko]) and np.array_equal(oid[kg], o.object_id[ko])
    fl = o.material[ko] == 1
    d = 0.02
    # the state is not at rest: pressure, wall contacts and a spread of densities
    assert float(o.pressure.max()) > 1000.0 and float(o.density[o.material == 1].max()) > 1010.0
    assert (o.x[ko][fl][:, 1] <= np.float32(0.04)).sum() > 1000
    got = {"dx_over_d": float(np.abs(x[kg] - o.x[ko]).max() / d),          # positions, in particle diameters
           "v": _maxrel(ps.v.to_numpy()[kg], o.v[ko]),
           "density": _maxrel(ps.density.to_numpy()[kg], o.density[ko]),
           "pressure": _maxrel(ps.pressure.to_numpy()[kg], o.pressure[ko]),   # (rho / rho0)^7 amplifies 7x
           "acceleration": _maxrel(ps.acceleration.to_numpy()[kg], o.acceleration[ko]),
           # same cell for (all but face-sitting) particles => both hold the same stable counting sort
           "cell_mismatch": float((ps.grid_ids.to_numpy()[kg] != o.grid_ids[ko]).mean())}
    tol = {"dx_over_d": 1e-4, "v": 1e-4, "density": REL, "pressure": 50 * REL, "acceleration": 50 * REL,
           "cell_mismatch": 1e-5}
    print("dragon_bath full size vs oracle:", got)
    assert all(got[k] < tol[k] for k in tol), (got, tol)


def test_stale_grid_is_refused():
    o, ps, solver = _pair(mixed_scene())
    solver.initialize()
    solver.compute_densities()
    solver.advect()
    with pytest.raises(RuntimeError, match="stale"):
        solver.compute_densities()


def test_out_of_grid_is_reported():
    o, ps, solver = _pair(mixed_scene())
    x = ps.x.to_numpy()
    x[0] = [-0.5, 0.1, 0.1]
    ps.x.from_numpy(x)
    ps.initialize_particle_system()
    with pytest.raises(RuntimeError, match="left the grid"):
        ps._engine.check_status()


def test_fused_step_fields_vs_oracle_and_overflow_path():
    """Fused production kernels (neighbour lists) per-field parity after ONE step, also on a state squeezed
    so hard that most particles exceed NBR_CAP = 96 neighbours (exercises the full-scan fallback)."""
    for squeeze, min_nbrs in ((1.0, 0), (0.6, 96)):
        sc = mixed_scene(with_dynamic=False)
        if min_nbrs:
            sc["Configuration"]["stiffness"] = 5  # rho ~ 3.7 rho0: keep (rho/rho0)^7 * k from ejecting the block
        o, ps, solver = _pair(sc, seed=11, amp=0.002)
        fl = o.material == 1
        c = o.x[fl].mean(axis=0)
        o.x[fl] = ((o.x[fl] - c) * np.float32(squeeze) + c).astype(np.float32)
        ps.x.from_numpy(o.x)
        o.initialize(); solver.initialize()
        o.step(); solver.step()
        assert np.array_equal(ps.x_0.to_numpy(), o.x_0)
        if min_nbrs:
            assert float(o.density[fl].max()) > 3200.0
            assert ps._engine.neighbor_stats()["overflow"] > 100
        assert _maxrel(ps.density.to_numpy(), o.density) < REL
        assert _maxrel(ps.pressure.to_numpy(), o.pressure) < 10 * REL
        assert _maxrel(ps.acceleration.to_numpy(), o.acceleration) < 10 * REL
        assert _maxrel(ps.v.to_numpy(), o.v) < 10 * REL
        assert _maxrel(ps.x.to_numpy(), o.x) < 1e-6


def _run_slab_check(nproc, extra=(), graph=False):
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = os.path.join(root, "tools", "check_slab_parity.py")
    if nproc == 1:
        cmd = [sys.executable, script, *extra]
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
               "--master-addr", "127.0.0.1", "--master-port", "29533", script, *extra]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, SPH_SHARD_GRAPH="1" if graph else "0"))
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert res.returncode == 0 and lines, res.stdout[-2000:] + res.stderr[-2000:]
    return json.loads(lines[-1])


def test_slab_mode_single_rank_equals_plain_engine():
    """Slab classification / trash bucket / info ranges with world = 1 (no exchange)."""
    out = _run_slab_check(1, ["--counts", "40", "16", "16", "--steps", "30"])
    assert out["ok"] and out["same_particle_set"] and out["max_dx_over_d"] < 1e-4


def test_slab_two_gpus_equals_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    for graph in (False, True):  # asynchronous launches (default) and CUDA-graph replay with the NCCL group captured
        out = _run_slab_check(2, ["--counts", "64", "24", "24", "--steps", "60"], graph=graph)
        assert out["ok"] and out["migrated"] and all(h > 0 for h in out["halo_bytes"]), (graph, out)


def test_armadillo_bath_dynamic_full_size():
    """BASELINE cfg 3 (1.74 M particles, three dynamic rigid bodies): a few real steps against the
    oracle, plus size-independent properties (rigidity of the shape-matched bodies, sortedness).

    The centre of mass of a body is an fp32 sum of 5490 same-sign terms; the oracle adds them
    serially (biased rounding, ~1e-4 m), the reference with unordered atomics, the engine with a
    fixed tree.  So the rigid particles are judged against the fp64 oracle, with the fp32 oracle's
    own distance to it as the noise floor."""
    from oracle.sph_oracle import OracleSim
    from sph_taichi_b200 import ParticleSystem, SimConfig, scene
    sc = scene.armadillo_bath_dynamic()
    ps = ParticleSystem(SimConfig(sc))
    assert ps.fluid_particle_num == 1723968 and ps.solid_particle_num == 3 * 5490
    solver = ps.build_solver()
    solver.initialize()
    o, o64 = OracleSim(sc), OracleSim(sc, f64=True)
    o.initialize(); o64.initialize()
    for oid in (1, 2, 3):
        assert _maxrel(ps.rigid_rest_cm[oid], o64.rest_cm[oid]) < 1e-6
    steps = 6
    solver.step(steps)
    for _ in range(steps):
        o.step(); o64.step()
    assert ps._engine.check_status() == 0
    x, x0, oid_g = ps.x.to_numpy(), ps.x_0.to_numpy(), ps.object_id.to_numpy()
    # rigid bodies share rest lattices (shifted copies), so key on (object id, x_0)
    kg = np.lexsort((x0[:, 2], x0[:, 1], x0[:, 0], oid_g))
    ko = np.lexsort((o.x_0[:, 2], o.x_0[:, 1], o.x_0[:, 0], o.object_id))
    x064 = o64.x_0.astype(np.float32)
    k64 = np.lexsort((x064[:, 2], x064[:, 1], x064[:, 0], o64.object_id))
    assert np.array_equal(x0[kg], o.x_0[ko]) and np.array_equal(oid_g[kg], o.object_id[ko])
    assert np.array_equal(x0[kg], x064[k64])
    fluid = oid_g[kg] == 0
    d = 0.02
    assert np.abs(x[kg] - o.x[ko])[fluid].max() / d < 1e-3
    err_rigid = np.abs(x[kg] - o64.x[k64])[~fluid].max() / d
    floor_rigid = np.abs(o.x[ko] - o64.x[k64])[~fluid].max() / d
    assert err_rigid < max(3 * floor_rigid, 1e-3), (err_rigid, floor_rigid)
    assert _maxrel(ps.v.to_numpy()[kg], o.v[ko]) < 1e-3
    assert np.all(np.diff(ps.grid_ids.to_numpy()) >= 0)
    for b in (1, 2, 3):  # shape matching keeps every body congruent to its rest shape
        sel = oid_g == b
        p, q = x[sel].astype(np.float64), x0[sel].astype(np.float64)
        dp = np.linalg.norm(p - p.mean(0), axis=1); dq = np.linalg.norm(q - q.mean(0), axis=1)
        assert np.abs(dp - dq).max() < 1e-4
        assert p[:, 1].mean() < q[:, 1].mean()  # and it is falling


def test_two_fluid_densities_take_the_general_force_kernel():
    """Two fluid blocks with different rest densities => non-uniform particle masses: the engine must drop
    the uniform-fluid packing (48 B/neighbour general kernel, separate advect) and still match the oracle."""
    from sph_taichi_b200 import scene
    sc = scene.dam_break_box([8, 10, 8], domain_end=[0.6, 0.6, 0.5], start=[0.06, 0.06, 0.06])
    second = dict(sc["FluidBlocks"][0])
    second.update({"objectId": 1, "start": [0.06 + 8 * 0.02, 0.06, 0.06], "end": [0.06 + 13.5 * 0.02, 0.06 + 9.5 * 0.02, 0.06 + 7.5 * 0.02],
                   "density": 800.0, "color": [200, 100, 50]})
    sc["FluidBlocks"].append(second)
    o, ps, solver = _pair(sc, seed=21, amp=0.002)
    o.initialize(); solver.initialize()
    steps = 20
    for _ in range(steps):
        o.step()
    solver.step(steps)
    assert len(np.unique(ps.m.to_numpy())) == 2
    ko, kg = order_by_x0(o.x_0), order_by_x0(ps.x_0.to_numpy())
    assert np.array_equal(ps.x_0.to_numpy()[kg], o.x_0[ko])
    assert np.abs(ps.x.to_numpy()[kg] - o.x[ko]).max() / 0.02 < 1e-3
    assert _maxrel(ps.density.to_numpy()[kg], o.density[ko]) < 1e-3


@pytest.mark.parametrize("seed,fill", [(21, 0.45), (22, 1.0)])
def test_random_scatter_state_vs_oracle(seed, fill):
    """Gas-like state: fluid particles scattered uniformly (about 1 per cell for fill = 0.45), so every kind
    of candidate range occurs -- empty columns next to full ones, odd and even starts, windows of a few
    particles -- next to a static block.  One fused step, field by field against the oracle."""
    sc = mixed_scene(fluid_counts=(14, 14, 14), with_dynamic=False)
    o, ps, solver = _pair(sc)
    rng = np.random.default_rng(seed)
    fl = o.material == 1
    lo, hi = np.float32(0.05), np.float32(0.05 + 0.5 * fill)
    o.x[fl] = rng.uniform(lo, hi, size=(int(fl.sum()), 3)).astype(np.float32)
    o.v[fl] = rng.uniform(-1, 1, size=(int(fl.sum()), 3)).astype(np.float32)
    ps.x.from_numpy(o.x)
    ps.v.from_numpy(o.v)
    o.initialize(); solver.initialize()
    assert np.array_equal(ps.grid_particles_num.to_numpy(), o.grid_particles_num)
    o.step(); solver.step()
    assert ps._engine.check_status() == 0
    assert np.array_equal(ps.x_0.to_numpy(), o.x_0)
    assert _maxrel(ps.density.to_numpy(), o.density) < REL
    assert _maxrel(ps.pressure.to_numpy(), o.pressure) < 10 * REL
    assert _maxrel(ps.acceleration.to_numpy(), o.acceleration) < 10 * REL
    assert _maxrel(ps.v.to_numpy(), o.v) < 10 * REL
    # close random pairs give accelerations of 1e5 m/s^2: the position error is dt times the velocity error
    dt = sc["Configuration"]["timeStepSize"]
    assert np.abs(ps.x.to_numpy() - o.x).max() <= dt * 10 * REL * float(np.abs(o.v).max()) + 1e-6


def test_emitter_adds_a_block_mid_run():
    """SURVEY section 8f rank 4 (the reference's planned emitter, particle_system.py:85-86): with
    `emitterReserve` a block is added through add_cube AFTER 12 steps; the run continues and matches an oracle
    that is handed the same 12-step state plus the same new block."""
    from oracle.sph_oracle import OracleSim
    from sph_taichi_b200 import ParticleSystem, SimConfig, scene
    d = 0.02
    base = scene.dam_break_box([10, 10, 10], domain_end=[0.8, 0.8, 0.6], start=[0.1, 0.06, 0.1])
    lower, size = np.array([0.42, 0.06, 0.1]), np.array([8 * d - 0.5 * d, 6 * d - 0.5 * d, 8 * d - 0.5 * d])
    sc = {k: (dict(v) if isinstance(v, dict) else list(v)) for k, v in base.items()}
    sc["Configuration"]["emitterReserve"] = 8 * 6 * 8
    ps = ParticleSystem(SimConfig(sc))
    assert ps.particle_max_num == 1000 + 384 and ps.particle_num[None] == 1000
    solver = ps.build_solver()
    solver.initialize()
    solver.step(12)
    ps.add_cube(object_id=0, lower_corner=lower, cube_size=size, material=1, is_dynamic=1, color=(50, 100, 200),
                density=1000.0, velocity=[0.0, -1.0, 0.0])
    assert ps.particle_num[None] == 1384 and ps.fluid_particle_num == 1384
    with pytest.raises(ValueError, match="emitterReserve"):
        ps.add_cube(object_id=0, lower_corner=lower, cube_size=size, material=1, is_dynamic=1)
    solver.step(12)
    assert ps._engine.check_status() == 0

    # oracle: the 1000-particle scene for 12 steps, then the same state + the new block in a 1384-particle oracle
    o1 = OracleSim(base)
    o1.initialize()
    for _ in range(12):
        o1.step()
    both = {k: (dict(v) if isinstance(v, dict) else list(v)) for k, v in base.items()}
    blk = dict(base["FluidBlocks"][0])
    blk.update(start=[float(v) for v in lower], end=[float(v) for v in lower + size], velocity=[0.0, -1.0, 0.0])
    both["FluidBlocks"] = [base["FluidBlocks"][0], blk]
    o2 = OracleSim(both)
    assert o2.n == 1384
    k1 = order_by_x0(o1.x_0)
    old = np.arange(1000)  # the first block's particles come first in the assembly order
    k2 = old[order_by_x0(o2.x_0[:1000])]
    assert np.array_equal(o2.x_0[k2], o1.x_0[k1])
    o2.x[k2] = o1.x[k1]; o2.v[k2] = o1.v[k1]
    for _ in range(12):
        o2.step()
    n = 1384
    x, x0 = ps.x.to_numpy()[:n], ps.x_0.to_numpy()[:n]
    kg, ko = order_by_x0(x0), order_by_x0(o2.x_0)
    assert np.array_equal(x0[kg], o2.x_0[ko])
    assert np.abs(x[kg] - o2.x[ko]).max() / d < 1e-4
    assert _maxrel(ps.v.to_numpy()[:n][kg], o2.v[ko]) < 1e-4
    assert _maxrel(ps.density.to_numpy()[:n][kg], o2.density[ko]) < 10 * REL
