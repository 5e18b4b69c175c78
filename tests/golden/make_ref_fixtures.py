#!/usr/bin/env python3
"""
tests/golden/make_ref_fixtures.py — what the REFERENCE's own kernels and scene loader (compiled for the CPU into
oracle/_ref by oracle/build_ref.py) compute for the configurations of tests/test_oracle_vs_ref.py and the reference
comparisons of tests/test_host.py, stored so that those tests run without the reference:

    python tests/golden/make_ref_fixtures.py --reference <reference checkout>

Writes into tests/golden/ref/:
  expected.json       per case: the per-bounce ray counters, and SHA-256 digests of primary-hit ids, radiance / AOV /
                      resolved bits (NaNs canonicalised as in tests.helpers.bits) or loaded scene arrays;
  libm_samples.npz    radiance of the reference kernels built with glibc's libm instead of include/rt_math.h, at a fixed
                      seeded sample of pixels;
  CornellBox.obj, ShaderBalls_faces.obj.xz, CornellBox_Dragon_faces.obj.xz, *.mtl
                      the reference's OBJ files (the two large ones shrunk by tests.ref_cases.obj_face_subset) and MTL files;
  checker3.jpg        the JPEG the reference ships with its assets;
  CGSkies_0036_rows.hdr.xz  every ENV_ROW_STEP-th scanline of the reference's environment map, bytes unchanged (the
                      run-length coding is per scanline), with the header's height adjusted.
The blue-noise cases run the reference kernels on tests.helpers.synthetic_sampler_tables(): the reference's own tables
are reference data and are not stored.
"""
import argparse
import json
import lzma
import os
import shutil
import sys
import tempfile

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)
from oracle import refbind  # noqa: E402
from raytracing_b200.camera import default_camera  # noqa: E402
from tests.helpers import digest, fuzz_configs, scene, synthetic_sampler_tables  # noqa: E402
from tests.ref_cases import (AOV_CAMERAS, BIT_EXACT, BLUE_NOISE, DEGENERATE, ENV_ROW_STEP, ENV_ROWS, LIBM, LIGHTS_LENS,  # noqa: E402
                             LOADER_SCENES, OUT, STATS, frame_key, libm_pixels, lights_lens_camera, loader_digests,
                             obj_face_subset, scene_arrays_digest, write_loader_input)

def _sample_record(r, mb, hits=True):
    rs = r.stats()
    rec = {k: rs[k][: mb + 1].tolist() for k in STATS}
    rec["radiance"] = digest(r.radiance()[..., :3])
    if hits:
        rec["primitive_id"] = digest(r.primary_hits()["primitive_id"])
    return rec


def _progressive(sc, cam, w, h, mb, samples, wf=False, blue_noise=False):
    from oracle.refbind import RefRenderer
    r = RefRenderer().open_arrays(sc)
    r.begin(w, h); r.set_camera(cam); r.set_max_bounces(mb); r.enable_white_furnace(wf)
    if blue_noise:
        r.set_blue_noise(True)
    out = []
    for _ in range(samples):
        r.integrate()
        out.append(_sample_record(r, mb))
    r.close()
    return out


def kernel_records():
    from oracle.refbind import RefRenderer
    from tests.scenes_extra import many_lights_scene, textured_cornell
    out = {}
    for name, w, h, mb, wf in BIT_EXACT:
        out["bit_exact/" + frame_key(name, w, h, mb, wf)] = _progressive(scene(name), default_camera(w, h), w, h, mb, 2, wf)
    for name, w, h, mb in LIGHTS_LENS:
        out["lights_lens/" + name] = _progressive(many_lights_scene(name), lights_lens_camera(w, h), w, h, mb, 2)
    for case, (name, w, h, mb, kw) in DEGENERATE.items():
        out["degenerate/" + case] = _progressive(scene(name), default_camera(w, h, **kw), w, h, mb, 2)
    for i, (name, w, h, mb, kw, wf) in enumerate(fuzz_configs()):
        out["fuzz/%d" % i] = _progressive(scene(name), default_camera(w, h, **kw), w, h, mb, 2, wf)
    refbind.set_sampler_tables(synthetic_sampler_tables())
    for name, w, h, mb, wf in BLUE_NOISE:
        out["blue_noise/" + frame_key(name, w, h, mb, wf)] = _progressive(scene(name), default_camera(w, h), w, h, mb, 3, wf, True)
    refbind.set_sampler_tables(None)
    w, h, mb = 96, 64, 4
    out["textured"] = _progressive(textured_cornell(), default_camera(w, h), w, h, mb, 1)[0]
    for name in ("CornellBox", "ShaderBalls"):
        w, h, mb = 128, 72, 3
        r = RefRenderer().open_arrays(scene(name)); r.begin(w, h)
        r.enable_denoiser(True); r.set_max_bounces(mb)
        frames = []
        for kw in AOV_CAMERAS:
            r.set_camera(default_camera(w, h, **kw)); r.integrate()
            frames.append({"albedo": digest(r.aov_albedo()[..., :3]), "depth": digest(r.aov_depth()), "normal": digest(r.aov_normal()[..., :3]),
                           "velocity": digest(r.aov_velocity()), "radiance": digest(r.radiance()[..., :3]), "resolved": digest(r.resolved())})
        r.close()
        out["aov/" + name] = frames
    samples = {}
    for name, w, h, mb, _ in LIBM:
        imgs = []
        for libm in (False, True):
            r = RefRenderer(libm=libm).open_arrays(scene(name))
            r.begin(w, h); r.set_camera(default_camera(w, h)); r.set_max_bounces(mb); r.integrate()
            imgs.append(r.radiance()[..., :3].copy()); r.close()
        out["libm/" + name] = {"radiance": digest(imgs[0])}
        samples[name] = imgs[1].reshape(-1, 3)[libm_pixels(w, h)]
    return out, samples


def host_records(reference):
    """The reference's own Scene + Bvh (+ kernels) on the generated inputs of tests/test_host.py."""
    from oracle.refbind import RefRenderer
    from tests import hdr_cases, obj_cases
    from tests.golden import make_texture_fixtures as mk
    from tests.golden.make_obj_fixtures import reference_env
    from tests.test_host import GENERATED_OBJ, LIVE_OBJ_CASES, numbers_obj, textured_obj_images, _textured_obj
    from raytracing_b200 import hostapi
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for seed in range(8):
            obj = obj_cases.write_case(os.path.join(tmp, "g%d" % seed), obj_cases.random_scene(200 + seed, GENERATED_OBJ[seed % 2]))
            w, h, mb = 96, 54, 5
            cam = hostapi.default_camera(w, h); cam["position"][:3] = (0.2, -3.4, 0.4)
            r = RefRenderer().open_obj(reference, obj)
            r.begin(w, h); r.set_camera(cam); r.set_max_bounces(mb); r.integrate()
            rec = _sample_record(r, mb)
            out["generated_obj/%d" % seed] = {"n_ext": rec["n_ext"], "primitive_id": rec["primitive_id"], "radiance": rec["radiance"]}
            r.close()
        live = {}
        for k, (seed, features) in enumerate(LIVE_OBJ_CASES):
            obj = obj_cases.write_case(os.path.join(tmp, "r%d" % k), obj_cases.random_scene(seed, features))
            live["%d_%s" % (seed, "_".join(features))] = scene_arrays_digest(RefRenderer().open_obj(reference, obj).scene())
        obj = obj_cases.write_case(os.path.join(tmp, "numbers"), numbers_obj())
        live["numbers"] = scene_arrays_digest(RefRenderer().open_obj(reference, obj).scene())
        for i, (name, data) in enumerate(hdr_cases.cases(seed=31).items()):
            root = os.path.join(tmp, "env%d" % i)
            os.mkdir(root)
            live["env/" + name] = hdr_cases.digest(*reference_env(root, data))
        out["obj_reader_live"] = live
        tex = os.path.join(tmp, "tex")
        os.mkdir(tex)
        obj = _textured_obj(__import__("pathlib").Path(tex), textured_obj_images(tex))
        g = RefRenderer().open_obj(reference, obj).scene()
        rec = {"textures": len(g["textures"]), "texels": digest(g["texels"]), "materials": digest(g["materials"]),
               "mtlIndex": digest(g["triangles"]["mtlIndex"])}
        rec.update({f: digest(g["textures"][f]) for f in ("width", "height", "data_start")})
        rec.update({v + ".texcoord": digest(g["triangles"][v]["texcoord"][:, :2]) for v in ("v1", "v2", "v3")})
        fresh = os.path.join(tmp, "fresh")
        names = mk.make_files(fresh, np.random.default_rng(77))
        rec["fresh"] = {n: [w, h, digest(t)] for n, (w, h, t) in mk.reference_texels(fresh, names).items()}
        rec["assets"] = {n: [w, h, digest(t)] for n, (w, h, t) in mk.reference_texels(OUT, ["checker3.jpg"]).items()}
        out["image_textures"] = rec
        for name in LOADER_SCENES:
            d = os.path.join(tmp, "loader_" + name)
            os.mkdir(d)
            out["loader/" + name] = loader_digests(RefRenderer().open_obj(reference, write_loader_input(name, d)).scene())
    return out


def store_env_rows(src, dst):
    """Every ENV_ROW_STEP-th scanline of a new-style run-length coded .hdr file, bytes unchanged."""
    data = open(src, "rb").read()
    head_end = data.index(b"\n\n") + 2
    res_end = data.index(b"\n", head_end) + 1
    h, w = (int(t) for t in data[head_end:res_end].split()[1::2])
    pos, rows = res_end, []
    for _ in range(h):
        start = pos
        assert data[pos:pos + 2] == b"\x02\x02" and (data[pos + 2] << 8 | data[pos + 3]) == w
        pos += 4
        for _c in range(4):
            x = 0
            while x < w:
                n = data[pos]
                if n > 128:
                    x, pos = x + n - 128, pos + 2
                else:
                    x, pos = x + n, pos + 1 + n
        rows.append(data[start:pos])
    keep = rows[::ENV_ROW_STEP]
    with lzma.open(dst, "wb", preset=9 | lzma.PRESET_EXTREME) as f:
        f.write(data[:head_end] + b"-Y %d +X %d\n" % (len(keep), w) + b"".join(keep))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="checkout of the reference project (oracle/_ref must be built from it)")
    a = ap.parse_args()
    os.makedirs(OUT, exist_ok=True)
    assets = os.path.join(a.reference, "assets")
    for name, stored in LOADER_SCENES.items():
        shutil.copyfile(os.path.join(assets, name + ".mtl"), os.path.join(OUT, name + ".mtl"))
        if stored.endswith(".xz"):
            with open(os.path.join(assets, name + ".obj")) as f, lzma.open(os.path.join(OUT, stored), "wt", preset=9 | lzma.PRESET_EXTREME) as g:
                g.write(obj_face_subset(f.read()))
        else:
            shutil.copyfile(os.path.join(assets, name + ".obj"), os.path.join(OUT, stored))
    shutil.copyfile(os.path.join(assets, "checker3.jpg"), os.path.join(OUT, "checker3.jpg"))
    store_env_rows(os.path.join(assets, "ibl", "CGSkies_0036_free.hdr"), ENV_ROWS)
    rec, samples = kernel_records()
    rec.update(host_records(a.reference))
    with open(os.path.join(OUT, "expected.json"), "w") as f:
        json.dump(rec, f, indent=0, sort_keys=True)
    np.savez_compressed(os.path.join(OUT, "libm_samples.npz"), **samples)
    print("wrote", len(rec), "records to", os.path.relpath(OUT, REPO))


if __name__ == "__main__":
    main()
