"""
tests/ref_cases.py — TEST INFRASTRUCTURE: the cases the reference comparisons run (tests/test_oracle_vs_ref.py, tests/test_host.py)
and the digests they compare, shared with tests/golden/make_ref_fixtures.py, which stores the reference's results for them
under tests/golden/ref.
"""
import lzma
import os
import shutil

import numpy as np

from raytracing_b200.camera import default_camera
from tests.helpers import digest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OUT = os.path.join(REPO, "tests", "golden", "ref")
ENV_ROWS = os.path.join(OUT, "CGSkies_0036_rows.hdr.xz")
STATS = ("n_ext", "n_miss", "n_hit", "n_shadow", "n_cont", "n_unoccluded")
ENV_ROW_STEP = 50

# (scene, width, height, max_bounces, white furnace)
BIT_EXACT = [("CornellBox", 97, 61, 3, False), ("CornellBox", 64, 64, 5, True), ("ShaderBalls", 160, 90, 8, False),
             ("CornellBox_Dragon", 120, 68, 6, False)]
BLUE_NOISE = [("CornellBox", 160, 136, 3, False),        # > 128 x 128: every tile pixel, incl. the ones whose ranking index runs past the table
              ("ShaderBalls", 144, 130, 8, False), ("CornellBox", 64, 64, 4, True)]
LIGHTS_LENS = [("CornellBox", 150, 90, 5), ("ShaderBalls", 128, 72, 4)]
DEGENERATE = {"zero_bounces": ("CornellBox", 96, 64, 0, {}),
              "all_miss": ("ShaderBalls", 80, 48, 4, {"position": (0.0, -30.0, 40.0), "pitch": 0.3}),
              "inside_geometry": ("ShaderBalls", 80, 48, 4, {"position": (0.0, 0.0, 0.35), "pitch": 1.9})}
# (scene, width, height, max_bounces, share of pixels allowed beyond 1e-4 relative)
LIBM = [("CornellBox", 160, 90, 8, 0.02), ("ShaderBalls", 160, 90, 8, 0.02), ("CornellBox_Dragon", 160, 90, 16, 0.04)]
LIBM_PIXELS = 512
AOV_CAMERAS = [{}, {"position": (0.05, -1.02, 1.01)}, {"position": (0.05, -1.02, 1.01)}]


def frame_key(name, w, h, mb, wf=False):
    return "%s_%dx%d_b%d%s" % (name, w, h, mb, "_wf" if wf else "")


def lights_lens_camera(w, h):
    return default_camera(w, h, position=(0.15, -1.3, 0.9), aperture=0.04, focus_distance=1.7)


def libm_pixels(w, h):
    return np.sort(np.random.default_rng(11).choice(w * h, LIBM_PIXELS, replace=False))


def scene_arrays_digest(a):
    """What tests/test_host.py compares of two loaders' scene arrays: vertex attributes, material index, packed materials,
    texture table (without its padding word, which the reference leaves uninitialised)."""
    parts = [a["triangles"][v][f][:, :3] for v in ("v1", "v2", "v3") for f in ("position", "texcoord", "normal")]
    parts += [a["triangles"]["mtlIndex"], a["materials"]] + [a["textures"][f] for f in ("width", "height", "data_start")]
    return digest(*parts)


# the loader / builder cases: the reference's OBJ files, whole when small, else one run of FACE_BLOCK consecutive faces in every
# FACE_STEP (runs of neighbouring faces share their vertex lines, which keeps the stored file small)
LOADER_SCENES = {"CornellBox": "CornellBox.obj", "ShaderBalls": "ShaderBalls_faces.obj.xz", "CornellBox_Dragon": "CornellBox_Dragon_faces.obj.xz"}
FACE_BLOCK, FACE_STEP = 64, 128


def obj_face_subset(text, block=FACE_BLOCK, step=FACE_STEP):
    """The faces of an OBJ text whose index // block is a multiple of step, with the position / texcoord / normal lines those
    faces use; every other line, and every kept line's text, unchanged except the renumbered indices of the faces."""
    lines = text.split("\n")
    faces = [i for i, ln in enumerate(lines) if ln.startswith("f ")]
    keep_faces = set(f for j, f in enumerate(faces) if (j // block) % step == 0)
    kinds = {"v": 0, "vt": 1, "vn": 2}
    used = [set(), set(), set()]
    for i in keep_faces:
        for tok in lines[i].split()[1:]:
            for k, ix in enumerate(tok.split("/")):
                if ix:
                    used[k].add(int(ix))
    count, new_index, out = [0, 0, 0], [{}, {}, {}], []
    for i, ln in enumerate(lines):
        head = ln.split(" ", 1)[0]
        if head in kinds:
            k = kinds[head]
            count[k] += 1
            if count[k] in used[k]:
                new_index[k][count[k]] = len(new_index[k]) + 1
                out.append(ln)
        elif head == "f":
            if i in keep_faces:
                toks = ["/".join(str(new_index[k][int(ix)]) if ix else "" for k, ix in enumerate(tok.split("/"))) for tok in ln.split()[1:]]
                out.append("f " + " ".join(toks) + (" " if ln.endswith(" ") else ""))
        else:
            out.append(ln)
    return "\n".join(out)


def loader_digests(a):
    """Per field, what the loader + BVH builder comparison checks of a scene: vertex attributes, material index, node boxes and
    records, packed materials, light origins, emissive list, scene info (the environment map is checked on its own)."""
    d = {v + "." + f: digest(a["triangles"][v][f][:, :3]) for v in ("v1", "v2", "v3") for f in ("position", "texcoord", "normal")}
    d["mtlIndex"] = digest(a["triangles"]["mtlIndex"])
    d.update({k: digest(a["nodes"][k][:, :3]) for k in ("bounds_min", "bounds_max")})
    d.update({k: digest(a["nodes"][k]) for k in ("offset", "num_primitives_axis")})
    d.update({"materials": digest(a["materials"]), "lights.origin": digest(a["lights"]["origin"][:, :3]), "emissive": digest(a["emissive"]),
              "scene_info": digest(a["scene_info"]), "counts": "%d triangles %d nodes" % (len(a["triangles"]), len(a["nodes"]))})
    return d


def write_loader_input(name, directory):
    """The OBJ of a loader case (decompressed) and the reference's MTL files, written into `directory`; returns the OBJ's path."""
    src = os.path.join(OUT, LOADER_SCENES[name])
    obj = os.path.join(str(directory), name + ".obj")
    with (lzma.open(src, "rb") if src.endswith(".xz") else open(src, "rb")) as f, open(obj, "wb") as g:
        g.write(f.read())
    for m in LOADER_SCENES:
        shutil.copyfile(os.path.join(OUT, m + ".mtl"), os.path.join(str(directory), m + ".mtl"))
    return obj


def write_env_rows(directory):
    """tests/golden/ref/CGSkies_0036_rows.hdr.xz decompressed into `directory`; returns the file's path."""
    path = os.path.join(str(directory), "CGSkies_0036_rows.hdr")
    with lzma.open(ENV_ROWS, "rb") as f, open(path, "wb") as g:
        g.write(f.read())
    return path
