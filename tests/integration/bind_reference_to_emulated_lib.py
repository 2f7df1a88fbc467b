"""INTEGRATION.md section 2, executed: the REFERENCE's ParticleSystem fields are bound to the C ABI of
include/sph_b200.h exactly as the stub in INTEGRATION.md does -- sph_create on a workspace, then per step
sph_pack(fields) / sph_step / sph_unpack(fields) on the field arrays -- and compared, step by step, with the
reference stepping itself.

Both sides come from tests/golden/ref_wcsph_binding.npz, written by tests/golden/make_reference_golden.py from the
reference's own source (run under the Taichi stand-in of tests/golden/ti_shim): its fields after
`solver.initialize()` are the bound arrays, and its state after every `solver.step()` is what they must track.

The library is the host-emulated build of the same sources (tests/emu/), so this runs without a GPU; "device
pointers" are host pointers.  Prints one JSON line.  TEST INFRASTRUCTURE.

    SPH_B200_LIB=tests/emu/_build/libsph_b200_emu.so python tests/integration/bind_reference_to_emulated_lib.py
"""
import ctypes as C
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

gold = np.load(os.path.join(ROOT, "tests", "golden", "ref_wcsph_binding.npz"))
scene = json.loads(str(gold["scene"]))
STEPS = int(gold["steps"])
FIELDS = ("object_id", "x", "x_0", "v", "acceleration", "m_V", "m", "density", "pressure", "material", "is_dynamic",
          "color", "grid_ids")
ps = {k: np.ascontiguousarray(gold["init_" + k]) for k in FIELDS}  # the reference's fields, bound below
twin = {k[5:]: gold[k] for k in gold.files if k.startswith("step_")}  # the reference's state after each step

# ---- the binding of INTEGRATION.md section 2 ----
from sph_taichi_b200 import _lib, engine  # noqa: E402  (parameter struct + argtypes only; no CUDA involved)

lib = _lib.load()
cfg = scene["Configuration"]
domain_size = [float(e) - float(s) for s, e in zip(cfg["domainStart"], cfg["domainEnd"])]
grid_num = np.ceil(np.array(domain_size) / (4.0 * cfg["particleRadius"])).astype(int)  # particle_system.py:44
params = engine.make_params(3, grid_num, cfg["particleRadius"], cfg["density0"], cfg["stiffness"], cfg["exponent"],
                            cfg["timeStepSize"], cfg["gravitation"], domain_size)
n = len(ps["x"])
n_solid = int((ps["material"] == 0).sum())
nbytes = lib.sph_workspace_bytes(C.byref(params), n, n_solid, 0)
ws = np.full(nbytes + 256, 0xAB, dtype=np.uint8)
base = (ws.ctypes.data + 255) // 256 * 256
ctx = C.c_void_p()
rc = lib.sph_create(C.byref(params), n, n_solid, 0, 0, C.c_void_p(base), nbytes, C.byref(ctx))
assert rc == 0, lib.sph_last_error(None)
solid_id = np.full(n, -1, np.int32)


def fields():
    f = _lib.SphFields()
    for k in FIELDS:
        a = ps[k]
        assert a.flags["C_CONTIGUOUS"]
        setattr(f, k, a.ctypes.data)
    f.solid_id = solid_id.ctypes.data
    return f


worst = {"x": 0.0, "v": 0.0, "density": 0.0}
same_order = True
for step in range(STEPS):
    solid = ps["material"] == 0
    solid_id[:] = -1
    solid_id[solid] = np.arange(int(solid.sum()), dtype=np.int32)
    fl = ps["material"] == 1
    assert lib.sph_set_solid_count(ctx, int(solid.sum()), 0) == 0
    assert lib.sph_set_fluid_uniform(ctx, 1, float(ps["m"][fl][0]), float(ps["m_V"][fl][0])) == 0
    f = fields()
    assert lib.sph_pack(ctx, C.byref(f), n, None) == 0, lib.sph_last_error(ctx)
    assert lib.sph_step(ctx, 1, None) == 0, lib.sph_last_error(ctx)
    assert lib.sph_unpack(ctx, C.byref(f), None) == 0, lib.sph_last_error(ctx)
    same_order &= bool(np.array_equal(ps["x_0"], twin["x_0"][step]))
    for k in worst:
        a, b = ps[k].astype(np.float64), twin[k][step].astype(np.float64)
        worst[k] = max(worst[k], float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)))
lib.sph_destroy(ctx)
print(json.dumps({"particles": int(n), "steps": STEPS, "same_particle_order": same_order, "max_rel_err": worst}))
