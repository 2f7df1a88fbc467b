"""INTEGRATION.md section 2 as an executable check: the fields of the reference's own ParticleSystem (stored from a
run under the Taichi stand-in) bound to the C ABI of the host-emulated library track the reference stepping itself."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_object_bound_to_the_c_abi_tracks_the_reference():
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_emu
    lib = build_emu.build()
    env = dict(os.environ, SPH_B200_LIB=lib)
    env.pop("SPH_EMU_LIB", None)
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "integration", "bind_reference_to_emulated_lib.py")],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert res.returncode == 0 and lines, res.stdout[-1500:] + res.stderr[-1500:]
    out = json.loads(lines[-1])
    assert out["same_particle_order"] and out["steps"] >= 5 and out["particles"] > 300
    assert out["max_rel_err"]["x"] < 1e-6 and out["max_rel_err"]["density"] < 2e-5 and out["max_rel_err"]["v"] < 1e-4
