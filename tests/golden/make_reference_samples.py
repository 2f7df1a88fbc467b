"""Data fixtures taken from the reference tree (erizmr/SPH_Taichi): its scene files, and a sample of its two meshes.

    python tests/golden/make_reference_samples.py REFERENCE_TREE

writes tests/golden/reference_scenes/*.json (byte copies of data/scenes/*.json) and
tests/golden/reference_models/<mesh>_sample.obj.  A mesh sample keeps SAMPLED_VERTICES vertices drawn with a fixed
seed, EVERY face that uses one of them, the vertices those faces also use, and the uv / normal records they
reference, as the original text; the sampled vertices come first in the file.  So for the sampled vertices the
(uv, normal) combinations a reader sees are exactly those of the full mesh (tests/test_voxelizer.py).
"""
import os
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SAMPLED_VERTICES = 32
MESHES = ("armadillo_small.obj", "Dragon_50k.obj")


def sample_obj(src, dst, k=SAMPLED_VERTICES, seed=0):
    recs = {"v": [], "vt": [], "vn": []}
    faces = []
    with open(src) as fh:
        for line in fh:
            tag = line.split(maxsplit=1)[0] if line.strip() else ""
            if tag in recs:
                recs[tag].append(line.rstrip("\n"))
            elif tag == "f":
                faces.append([tok.split("/") for tok in line.split()[1:]])
    nv = len(recs["v"])

    def index(tok, n):
        i = int(tok)
        return i - 1 if i > 0 else n + i

    chosen = sorted(np.random.default_rng(seed).choice(nv, k, replace=False).tolist())
    pick = set(chosen)
    kept = [f for f in faces if any(index(c[0], nv) in pick for c in f)]
    used = {"v": list(chosen), "vt": [], "vn": []}
    for f in kept:
        for c in f:
            for slot, tag in enumerate(("v", "vt", "vn")):
                if len(c) > slot and c[slot]:
                    used[tag].append(index(c[slot], len(recs[tag])))
    remap = {tag: {old: new + 1 for new, old in enumerate(dict.fromkeys(used[tag]))} for tag in used}
    with open(dst, "w") as out:
        out.write(f"# sample of {os.path.basename(src)}: its first {k} vertices with every face that uses them\n")
        for tag in ("v", "vt", "vn"):
            for old in remap[tag]:
                out.write(recs[tag][old] + "\n")
        for f in kept:
            toks = []
            for c in f:
                toks.append("/".join("" if not t else str(remap[tag][index(t, len(recs[tag]))])
                                     for t, tag in zip(c, ("v", "vt", "vn"))))
            out.write("f " + " ".join(toks) + "\n")


if __name__ == "__main__":
    ref = sys.argv[1]
    scenes = os.path.join(HERE, "reference_scenes")
    os.makedirs(scenes, exist_ok=True)
    for f in sorted(os.listdir(os.path.join(ref, "data", "scenes"))):
        if f.endswith(".json"):
            shutil.copyfile(os.path.join(ref, "data", "scenes", f), os.path.join(scenes, f))
    models = os.path.join(HERE, "reference_models")
    os.makedirs(models, exist_ok=True)
    for name in MESHES:
        sample_obj(os.path.join(ref, "data", "models", name), os.path.join(models, name[:-4] + "_sample.obj"))
