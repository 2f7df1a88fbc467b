"""Golden vectors from the REFERENCE'S OWN SOURCE (erizmr/SPH_Taichi, /root/reference), executed under the
pure-Python Taichi stand-in in tests/golden/ti_shim/ (see its docstring for the semantics it implements).

    python tests/golden/make_reference_golden.py          # writes tests/golden/ref_*.npz (+ ref_*_body*.npz)

The reference files particle_system.py / sph_base.py / WCSPH.py / DFSPH.py / config_builder.py are imported
unmodified; nothing of them is copied into this repository.  Each golden file holds the scene (JSON), the number
of steps, and the particle fields after `solver.initialize()` and after the last `solver.step()`, in the
reference's own particle order.  tests/test_golden_reference.py replays the scenes with the CPU oracle.
This script cannot run on the GPU box (no reference tree there); the vectors are committed.
"""
import contextlib
import io
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("SPH_REFERENCE", "/root/reference")


def base_cfg(method=0, dt=0.0004, domain=(0.6, 0.6, 0.6)):
    return {"domainStart": [0.0, 0.0, 0.0], "domainEnd": list(domain), "particleRadius": 0.01,
            "numberOfStepsPerRenderUpdate": 1, "density0": 1000, "simulationMethod": method,
            "gravitation": [0.0, -9.81, 0.0], "timeStepSize": dt, "stiffness": 50000, "exponent": 7,
            "boundaryHandlingMethod": 0, "exportFrame": False, "exportPly": False, "exportObj": False}


def fluid(start, counts, velocity=(0.0, 0.0, 0.0), oid=0):
    d = 0.02
    end = [start[k] + (counts[k] - 0.5) * d for k in range(3)]
    return {"objectId": oid, "start": list(start), "end": end, "translation": [0.0, 0.0, 0.0], "scale": [1, 1, 1],
            "velocity": list(velocity), "density": 1000.0, "color": [50, 100, 200]}


def block(oid, start, counts, dynamic, velocity=(0.0, 0.0, 0.0), density=1000.0):
    b = fluid(start, counts, velocity, oid)
    b.update({"isDynamic": bool(dynamic), "density": density, "color": [255, 255, 255]})
    return b


def body(oid, counts, offset, dynamic, velocity=(0.0, 0.0, 0.0), density=800.0):
    spec = "lattice:" + ",".join(str(int(v)) for v in list(counts) + list(offset))
    return {"objectId": oid, "geometryFile": spec, "translation": [0.0, 0.0, 0.0], "rotationAxis": [0, 1, 0],
            "rotationAngle": 0, "scale": [1, 1, 1], "velocity": list(velocity), "density": density,
            "color": [255, 255, 255], "isDynamic": bool(dynamic)}


SCENES = {
    # fluid next to a static and under a falling dynamic RigidBlock: Akinci volumes, fluid-solid coupling, reactions
    "wcsph_blocks": (dict(Configuration=base_cfg(),
                          FluidBlocks=[fluid([0.10, 0.06, 0.10], (7, 8, 7), (0.3, -1.0, 0.0))],
                          RigidBlocks=[block(1, [0.24, 0.06, 0.10], (3, 6, 6), False),
                                       block(2, [0.10, 0.23, 0.10], (4, 3, 4), True, (0.0, -0.5, 0.0), 600.0)]), 8),
    # fast block into the -y floor, the +x and the -z walls: clamp + reflection on low and high walls
    "wcsph_walls": (dict(Configuration=base_cfg(),
                         FluidBlocks=[fluid([0.455, 0.05, 0.05], (6, 7, 6), (4.0, -3.0, -2.5))]), 12),
    # rigid BODIES (shape matching, rest centre of mass, boundary clamp of solids) through the trimesh stand-in
    "wcsph_bodies": (dict(Configuration=base_cfg(),
                          FluidBlocks=[fluid([0.10, 0.06, 0.10], (6, 7, 6), (0.0, -1.0, 0.0))],
                          RigidBodies=[body(1, (4, 4, 4), (6, 11, 6), True, (0.5, -2.0, 0.0), 700.0),
                                       body(2, (3, 5, 6), (12, 3, 5), False)]), 7),
    # the 1 200-particle dam break of tests/golden/dam_break_*: 40 steps, two wall contacts, an evolving free surface
    "wcsph_dambreak": (dict(Configuration=base_cfg(domain=(0.8, 0.6, 0.4)),
                            FluidBlocks=[fluid([0.05, 0.05, 0.05], (10, 12, 10), (0.0, 0.0, 0.0))]), 40),
    # BASELINE configs[0]: the 8 K cube (20^3 lattice in the unit box) -- about 80 s per step in pure Python, so only
    # a few steps; only x_0 / x / v / density of the final state are kept (SMALL below)
    "wcsph_cube8k": (dict(Configuration=base_cfg(domain=(1.0, 1.0, 1.0)),
                          FluidBlocks=[dict(fluid([0.1, 0.1, 0.1], (20, 20, 20)), end=[0.49, 0.49, 0.49])]), 6),
    # DFSPH (divergence + pressure solver loops of the reference, host-side convergence tests)
    "dfsph_blocks": (dict(Configuration=base_cfg(method=4, dt=0.004),
                          FluidBlocks=[fluid([0.10, 0.06, 0.10], (5, 7, 6), (2.0, -1.0, 0.0)),
                                       fluid([0.21, 0.06, 0.10], (5, 7, 6), (-2.0, -1.0, 0.0), oid=3)],
                          RigidBlocks=[block(1, [0.32, 0.06, 0.10], (3, 5, 6), False)]), 4),
    # DFSPH with a dynamic RigidBlock: the reaction terms of the solver sweeps on dynamic solid particles
    "dfsph_dynamic_block": (dict(Configuration=base_cfg(method=4, dt=0.004),
                                 FluidBlocks=[fluid([0.10, 0.06, 0.10], (6, 6, 6), (0.0, -1.5, 0.0))],
                                 RigidBlocks=[block(1, [0.12, 0.19, 0.12], (4, 3, 4), True, (0.0, -2.5, 0.0), 500.0)]), 3),
    # DFSPH with a shape-matched rigid BODY (the situation of the reference's dragon_bath_dynamic_dfsph.json)
    "dfsph_bodies": (dict(Configuration=base_cfg(method=4, dt=0.004),
                          FluidBlocks=[fluid([0.10, 0.06, 0.10], (6, 6, 6), (0.0, -1.0, 0.0))],
                          RigidBodies=[body(1, (4, 3, 4), (6, 10, 6), True, (0.3, -2.0, 0.0), 600.0)]), 3),
    # the scene tests/integration/bind_reference_to_emulated_lib.py replays through the C ABI (TRAJECTORY below)
    "wcsph_binding": (dict(Configuration=base_cfg(),
                           FluidBlocks=[fluid([0.10, 0.06, 0.10], (6, 7, 6), (0.5, -1.0, 0.0))],
                           RigidBlocks=[block(1, [0.23, 0.06, 0.10], (3, 5, 6), False)]), 6),
}
SMALL = ("wcsph_cube8k",)
# these also keep the initial colours and x_0 / x / v / density after EVERY step (step_* arrays, one row per step)
TRAJECTORY = ("wcsph_binding",)
STEP_FIELDS = ("x_0", "x", "v", "density")
FIELDS = ("object_id", "x_0", "x", "v", "acceleration", "m_V", "m", "density", "pressure", "material", "is_dynamic",
          "grid_ids")


def snapshot(ps, prefix, out):
    for f in FIELDS:
        out[prefix + f] = getattr(ps, f).to_numpy()
    out[prefix + "grid_particles_num"] = ps.grid_particles_num.to_numpy()
    if ps.simulation_method == 4:
        out[prefix + "dfsph_factor"] = ps.dfsph_factor.to_numpy()
        out[prefix + "density_adv"] = ps.density_adv.to_numpy()


def run_reference(scene, steps, allow_oob=False, trajectory=False):
    sys.path.insert(0, os.path.join(HERE, "ti_shim"))
    sys.path.insert(0, REF)
    import taichi as ti
    from config_builder import SimConfig
    from particle_system import ParticleSystem
    fd, path = tempfile.mkstemp(suffix=".json")
    os.write(fd, json.dumps(scene).encode())
    os.close(fd)
    out = {}
    log = io.StringIO()
    with contextlib.redirect_stdout(log):
        ps = ParticleSystem(SimConfig(scene_file_path=path), GGUI=False)
        # compile-time constants of the reference's kernels are Python floats (weakly typed), not numpy float64
        ps.domain_size = [float(v) for v in ps.domain_size]
        solver = ps.build_solver()
        solver.initialize()
        snapshot(ps, "init_", out)
        if trajectory:
            out["init_color"] = ps.color.to_numpy()
        per_step = {f: [] for f in STEP_FIELDS}
        for _ in range(steps):
            solver.step()
            if trajectory:
                for f in STEP_FIELDS:
                    per_step[f].append(getattr(ps, f).to_numpy())
        snapshot(ps, "final_", out)
        if trajectory:
            out.update({"step_" + f: np.stack(v) for f, v in per_step.items()})
    os.unlink(path)
    # Particles resting on an UPPER wall sit in the last cell layer, whose +1 neighbours lie outside the grid: the
    # reference reads them unchecked (SURVEY Q3; harmless on Taichi only because the adjacent memory holds zeros).
    # The stand-in reads such cells as empty -- what the oracle and the engine do by skipping them -- and counts them.
    assert allow_oob or ti.oob_reads == 0, f"{ti.oob_reads} reads of neighbour cells outside the grid"
    out["oob_cell_reads"] = np.array(ti.oob_reads)
    ti.oob_reads = 0
    # the reference prints its loop counts: "DFSPH - iteration V: n ..." and "DFSPH - iterations: n ..." per step
    import re
    out["dfsph_iterations_v"] = np.array([int(v) for v in re.findall(r"DFSPH - iteration V: (\d+)", log.getvalue())])
    out["dfsph_iterations"] = np.array([int(v) for v in re.findall(r"DFSPH - iterations: (\d+)", log.getvalue())])
    return out


if __name__ == "__main__":
    out_dir = HERE
    args = sys.argv[1:]
    if args[:1] == ["--out"]:
        out_dir, args = args[1], args[2:]
    names = args or list(SCENES)
    for name in names:
        scene, steps = SCENES[name]
        out = run_reference(json.loads(json.dumps(scene)), steps, allow_oob=(name in ("wcsph_walls", "wcsph_dambreak")),
                            trajectory=name in TRAJECTORY)
        # the oracle / engine side reads rigid bodies from a lattice fixture instead of a mesh
        mine = json.loads(json.dumps(scene))
        for k, b in enumerate(mine.get("RigidBodies", [])):
            v = [int(t) for t in b["geometryFile"].split(":", 1)[1].split(",")]
            g = np.stack(np.meshgrid(*[np.arange(c) for c in v[:3]], indexing="ij"), -1).reshape(-1, 3) + np.array(v[3:6])
            fix = f"ref_{name}_body{b['objectId']}.npz"
            np.savez_compressed(os.path.join(out_dir, fix), pitch=np.float64(0.02), lattice=g.astype(np.int64))
            b["geometryFile"] = "(synthetic lattice block)"
            b["voxelizedPointsFile"] = fix
        if name in SMALL:  # keep the committed file small: final state only, the fields a trajectory pin needs
            keep = ("final_object_id", "final_x_0", "final_x", "final_v", "final_density", "final_grid_ids",
                    "final_grid_particles_num", "oob_cell_reads", "dfsph_iterations_v", "dfsph_iterations")
            out = {k: v for k, v in out.items() if k in keep}
        np.savez_compressed(os.path.join(out_dir, f"ref_{name}.npz"), scene=json.dumps(mine), steps=steps, **out)
        print(name, "particles", len(out["final_x"]), "steps", steps)
