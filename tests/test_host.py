"""
Host-side C++ (raytracing_b200/host: Scene loader, SAH BVH builder, HDR reader, Integrator mirror,
CUDAPathTraceIntegrator, headless Render).  CPU tests run everywhere; the Render tests need a GPU.
"""
import os

import numpy as np
import pytest

from oracle.orcbind import Oracle
from raytracing_b200 import hostapi, scene_io
from raytracing_b200.camera import default_camera
from tests.helpers import bits, digest, scene, synthetic_sampler_tables

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROC_OBJ = os.path.join(REPO, "tests", "golden", "scenes", "procedural.obj")
REF_GOLDEN = os.path.join(REPO, "tests", "golden", "ref")          # what the reference made of the inputs below (make_ref_fixtures.py)


def reference_record(key):
    import json
    with open(os.path.join(REF_GOLDEN, "expected.json")) as f:
        return json.load(f)[key]


def write_hdr(path, rgbe, rle=True):
    """Minimal Radiance .hdr writer (new-style RLE scanlines of literal chunks, or flat pixels)."""
    h, w, _ = rgbe.shape
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n")
        f.write(f"-Y {h} +X {w}\n".encode())
        for y in range(h):
            if rle and 8 <= w <= 32767:
                f.write(bytes([2, 2, w >> 8, w & 255]))
                for c in range(4):
                    x = 0
                    while x < w:
                        n = min(128, w - x)
                        if n >= 3 and (x // 128) % 2 == 1:      # alternate: a run of the first value, then literals
                            f.write(bytes([128 + 2, int(rgbe[y, x, c])]))
                            row = rgbe[y, x:x + 2, c].copy(); row[:] = rgbe[y, x, c]
                            rgbe[y, x:x + 2, c] = row
                            x += 2
                            continue
                        f.write(bytes([n])); f.write(rgbe[y, x:x + n, c].astype(np.uint8).tobytes())
                        x += n
            else:
                f.write(rgbe[y].astype(np.uint8).tobytes())
    return rgbe


def decode_rgbe(rgbe):
    """hdr_loader.cpp:102-120: (mantissa / 256) * 2^(E - 128), alpha 0."""
    e = rgbe[..., 3].astype(np.int32) - 128
    d = np.ldexp(np.float32(1.0), e).astype(np.float32)
    out = np.zeros(rgbe.shape[:2] + (4,), dtype=np.float32)
    for c in range(3):
        out[..., c] = (rgbe[..., c].astype(np.float32) / np.float32(256.0)) * d
    return out


def make_env(tmp_path, w=48, h=24, rle=True):
    rng = np.random.default_rng(3)
    rgbe = rng.integers(0, 256, size=(h, w, 4)).astype(np.int64)
    rgbe[..., 3] = rng.integers(120, 134, size=(h, w))
    path = str(tmp_path / f"env_{w}x{h}_{int(rle)}.hdr")
    rgbe = write_hdr(path, rgbe, rle)
    return path, decode_rgbe(rgbe)


def test_default_camera_matches_python_mirror():
    for (w, h) in [(1920, 1080), (256, 256), (3840, 2160), (333, 127)]:
        assert hostapi.default_camera(w, h).tobytes() == default_camera(w, h).tobytes()


@pytest.mark.parametrize("w,rle", [(48, True), (300, True), (5, False), (48, False)])
def test_hdr_reader(tmp_path, w, rle):
    path, expect = make_env(tmp_path, w=w, h=7, rle=rle)
    s = hostapi.HostScene(PROC_OBJ)
    s.add_directional_light((0, 0, 1), (1, 1, 1))
    s.finalize(env_path=path)
    a = s.arrays()
    assert (a["env_width"], a["env_height"]) == (w, 7)
    assert np.array_equal(bits(a["env"].reshape(7, w, 4)), bits(expect))
    s.close()


def test_procedural_obj_loads_and_bvh_is_a_valid_tree():
    s = hostapi.HostScene(PROC_OBJ)
    s.add_directional_light((-0.6, -1.5, 3.5), (15, 10, 5))
    s.build_bvh()
    s.finalize(env=np.zeros(4, dtype=np.float32), env_width=1, env_height=1)
    a = s.arrays()
    tris, nodes = a["triangles"], a["nodes"]
    assert len(tris) == 458 and len(a["materials"]) == 7 and len(a["lights"]) == 1
    assert a["scene_info"]["analytic_light_count"][0] == 1 and a["scene_info"]["emissive_count"][0] == 2 == len(a["emissive"])
    # directional light is normalised (scene.cpp:347-351)
    assert abs(np.linalg.norm(a["lights"]["origin"][0, :3]) - 1) < 1e-6
    # every triangle is covered by exactly one leaf, child boxes are inside parents, leaves hold <= 4 prims
    count = nodes["num_primitives_axis"] >> 16
    leaves = count > 0
    cover = np.zeros(len(tris), dtype=int)
    for off, c in zip(nodes["offset"][leaves], count[leaves]):
        cover[off:off + c] += 1
    assert (cover == 1).all() and count.max() <= 4
    for i in np.nonzero(~leaves)[0]:
        for child in (i + 1, nodes["offset"][i]):
            assert (nodes["bounds_min"][child, :3] >= nodes["bounds_min"][i, :3]).all()
            assert (nodes["bounds_max"][child, :3] <= nodes["bounds_max"][i, :3]).all()
    # materials: the Tf 0 sheet is pass-through, the lamp is emissive, roughness/metalness are 8-bit packed
    mats = a["materials"]
    assert ((mats["ior_emission_idx_transparency"] >> 16) & 0xFF).min() == 0
    assert (mats["emission"] != 0).sum() == 1
    s.close()


def _pack_like_stb(img):
    """PIL image -> the reference's texel words the way LoadSTB builds them from stb_image's channel count
    (image_loader.cpp:30-63): L -> (y,0,0,0), LA -> (y,a,0,0), RGB -> (r,g,b,0), RGBA -> (r,g,b,a); 16-bit -> high byte."""
    a = np.asarray(img)
    if a.dtype == np.uint16 or a.dtype == np.int32:
        a = (a.astype(np.uint32) >> 8).astype(np.uint8)
    if a.ndim == 2:
        a = a[..., None]
    c = a.shape[2]
    w = a[..., 0].astype(np.uint32)
    for k in range(1, c):
        w |= a[..., k].astype(np.uint32) << (8 * k)
    return w.reshape(-1)


def _textured_obj(tmp_path, files):
    """A quad (two triangles, uv 0..1) per texture file, one material each, every map_* key in use."""
    keys = ["map_Kd", "map_Ks", "map_Pr", "map_Pm", "map_Ke", "map_d"]
    with open(tmp_path / "tex.mtl", "w") as f:
        for i, name in enumerate(files):
            f.write(f"newmtl m{i}\nKd 0.5 0.5 0.5\nKs 0.5 0.5 0.5\nKe 0.2 0.2 0.2\nTf 1 1 1\nPr 0.5\n{keys[i % len(keys)]} -s 1 1 1 {name}\n")
            if i == 0:
                f.write(f"map_Ks {files[-1]}\n")               # the same file twice: cached, one texture
    with open(tmp_path / "tex.obj", "w") as f:
        f.write("mtllib tex.mtl\nvn 0 0 1\nvt 0 0\nvt 1 0\nvt 1 1\nvt 0 1\n")
        for i in range(len(files)):
            x = 1.5 * i
            f.write(f"v {x} 0 0\nv {x + 1} 0 0\nv {x + 1} 1 0\nv {x} 1 0\nusemtl m{i}\n")
            b = 4 * i
            f.write(f"f {b + 1}/1/1 {b + 2}/2/1 {b + 3}/3/1\nf {b + 1}/1/1 {b + 3}/3/1 {b + 4}/4/1\n")
    return str(tmp_path / "tex.obj")


def test_image_textures_png_tga(tmp_path):
    """map_* textures (SURVEY 8f row 3): PNG (grey 1/8/16 bit, grey+alpha, RGB, RGBA, palette with and without tRNS, every row
    filter) and TGA (24/32 bit, grey, RLE, both row orders) decoded by host/image_loader.cpp into the reference's texel words,
    checked against PIL's decode packed like LoadSTB; texture indices in the order scene.cpp:155-186 loads them; same file -> one
    texture; an arithmetic-coded JPEG fails loudly."""
    from PIL import Image
    rng = np.random.default_rng(5)
    imgs = {}

    def rnd(shape, dtype=np.uint8, hi=256):
        return rng.integers(0, hi, size=shape).astype(dtype)
    imgs["rgb.png"] = Image.fromarray(rnd((13, 17, 3)), "RGB")
    imgs["rgba.png"] = Image.fromarray(rnd((9, 31, 4)), "RGBA")
    imgs["grey.png"] = Image.fromarray(rnd((7, 5)), "L")
    imgs["la.png"] = Image.fromarray(rnd((6, 6, 2)), "LA")
    imgs["grey16.png"] = Image.fromarray(rnd((5, 9), np.uint16, 65536))
    imgs["bits1.png"] = Image.fromarray(rnd((11, 19), hi=2) * 255, "L").convert("1")
    pal = Image.fromarray(rnd((10, 12), hi=16), "P"); pal.putpalette(list(rnd(48)))
    imgs["pal.png"] = pal
    imgs["rgb.tga"] = Image.fromarray(rnd((8, 14, 3)), "RGB")
    imgs["rgba_rle.tga"] = Image.fromarray(np.repeat(rnd((6, 5, 4)), 4, axis=1), "RGBA")     # runs: RLE packets of both kinds
    imgs["grey.tga"] = Image.fromarray(rnd((4, 7)), "L")
    expect = {}
    for name, im in imgs.items():
        path = str(tmp_path / name)
        if name == "rgba_rle.tga":
            im.save(path, compression="tga_rle")
        elif name == "rgb.tga":
            im.save(path, orientation=1)             # top-left origin; the default writer stores bottom-up
        else:
            im.save(path)
        back = Image.open(path)
        if name == "bits1.png":
            expect[name] = _pack_like_stb(back.convert("L"))
        elif name == "pal.png":
            expect[name] = _pack_like_stb(back.convert("RGB"))
        else:
            expect[name] = _pack_like_stb(back)
    files = list(imgs)
    s = hostapi.HostScene(_textured_obj(tmp_path, files))
    s.add_directional_light((0, 0, 1), (1, 1, 1))
    s.finalize(env=np.zeros(4, dtype=np.float32), env_width=1, env_height=1)
    a = s.arrays()
    # load order: material 0 loads its map_Kd (files[0]) then its map_Ks (files[-1]); the others follow, files[-1] is cached
    order = [files[0], files[-1]] + files[1:-1]
    assert len(a["textures"]) == len(files)
    for idx, name in enumerate(order):
        t = a["textures"][idx]
        w, h = imgs[name].size
        assert (t["width"], t["height"]) == (w, h), name
        got = a["texels"][t["data_start"]: t["data_start"] + w * h]
        assert np.array_equal(got, expect[name]), name
    m = a["materials"]
    tex_of = {name: i for i, name in enumerate(order)}
    assert m["diffuse_albedo"][0] >> 24 == tex_of[files[0]] and m["specular_albedo"][0] >> 24 == tex_of[files[-1]]
    assert (m["specular_albedo"][1] >> 24) == tex_of[files[1]]                       # material 1: map_Ks
    assert ((m["roughness_metalness"][2] >> 8) & 0xFF) == tex_of[files[2]]           # material 2: map_Pr
    assert (m["roughness_metalness"][3] >> 24) == tex_of[files[3]]                   # material 3: map_Pm
    assert ((m["ior_emission_idx_transparency"][4] >> 8) & 0xFF) == tex_of[files[4]] # material 4: map_Ke
    assert (m["ior_emission_idx_transparency"][5] >> 24) == tex_of[files[5]]         # material 5: map_d
    assert (m["diffuse_albedo"][1] >> 24) == 0xFF                                    # no diffuse texture there
    s.close()
    with open(tmp_path / "x.jpg", "wb") as f:                        # start-of-image, then nothing a decoder can use
        f.write(b"\xff\xd8\xff\xc9\x00\x04\x00\x00\xff\xd9")
    with pytest.raises(hostapi.HostError, match="JPEG"):
        hostapi.HostScene(_textured_obj(tmp_path, ["x.jpg"]))


def _scene_arrays_from_obj(obj_path, scale=1.0, flip_yz=False):
    s = hostapi.HostScene(obj_path, scale=scale, flip_yz=flip_yz)
    s.add_directional_light((-0.6, -1.5, 3.5), (15, 10, 5))
    s.build_bvh()
    s.finalize(env=np.zeros(4, dtype=np.float32), env_width=1, env_height=1)
    a = s.arrays()
    s.close()
    return a


def _same_scene_arrays(a, g):
    """None, or what differs between the loader's arrays `a` and the reference's `g` (triangles, materials, texture table)."""
    if len(a["triangles"]) != len(g["triangles"]):
        return "triangle count %d, expected %d" % (len(a["triangles"]), len(g["triangles"]))
    for v in ("v1", "v2", "v3"):
        for f in ("position", "texcoord", "normal"):
            if not np.array_equal(bits(a["triangles"][v][f][:, :3]), bits(g["triangles"][v][f][:, :3])):
                return v + "." + f
    if not np.array_equal(a["triangles"]["mtlIndex"], g["triangles"]["mtlIndex"]):
        return "mtlIndex"
    if a["materials"].tobytes() != g["materials"].tobytes():
        return "materials"
    for f in ("width", "height", "data_start"):
        if not np.array_equal(a["textures"][f], g["textures"][f]):
            return "textures." + f
    return None


def test_obj_reader_cases_load_like_the_reference(tmp_path):
    """host/obj_reader.cpp on the inputs of tests/obj_cases.py — number syntax and rounding, material-name tokenising, texture
    options, dropped faces, quad diagonals, ear clipping of concave polygons, line ends ..., 30 generated scenes, the --scale and
    --flip_yz load options — against what
    the reference's own loader (tinyobjloader + Scene::Load + Bvh::BuildCPU) made of the same files
    (tests/golden/make_obj_fixtures.py)."""
    from tests import obj_cases
    from tests.golden.make_obj_fixtures import all_cases, LOAD_OPTIONS
    expected = np.load(os.path.join(REPO, "tests", "golden", "obj", "expected.npz"))
    n = 0
    for name, files in all_cases():
        a = _scene_arrays_from_obj(obj_cases.write_case(str(tmp_path / name), files), *LOAD_OPTIONS.get(name, (1.0, False)))
        g = {k: expected[name + ":" + k] for k in ("triangles", "materials", "textures")}
        assert _same_scene_arrays(a, g) is None, (name, _same_scene_arrays(a, g))
        n += 1
    assert n >= 60
    # the number reader on its own: digit accumulation, not strtod
    assert hostapi.obj_parse_number("1.9662156701087952") == 1.9662156701087954 != float("1.9662156701087952")
    assert hostapi.obj_parse_number("1.5x") == 1.5 and hostapi.obj_parse_number("-.25") == -0.25 and hostapi.obj_parse_number("5.") == 5.0
    assert hostapi.obj_parse_number("1e") is None and hostapi.obj_parse_number("abc") is None and hostapi.obj_parse_number("-") is None
    assert hostapi.obj_parse_number("1.5e+1") == 15.0 and hostapi.obj_parse_number("1E-2") == 0.01


def _load_env(path):
    s = hostapi.HostScene(PROC_OBJ)
    s.add_directional_light((0, 0, 1), (1, 1, 1))
    s.finalize(env_path=path)
    a = s.arrays()
    s.close()
    return a["env"], int(a["env_width"]), int(a["env_height"])


def test_hdr_reader_cases_load_like_the_reference(tmp_path):
    """LoadHDR on the files of tests/hdr_cases.py (flat / new / old run-length coding, window edges of the new coding, two repeat
    markers in a row — where the reference keeps the count in 8 bits —, look-alike scanline starts, a file cut short) against
    digests of what the reference's LoadHDR read (tests/golden/make_obj_fixtures.py)."""
    import json
    from tests import hdr_cases
    with open(os.path.join(REPO, "tests", "golden", "obj", "hdr_files.json")) as f:
        expected = json.load(f)
    files = hdr_cases.cases()
    assert set(files) == set(expected) and len(files) >= 20
    for name, data in files.items():
        with open(tmp_path / "e.hdr", "wb") as f:
            f.write(data)
        assert hdr_cases.digest(*_load_env(str(tmp_path / "e.hdr"))) == expected[name], name


GENERATED_OBJ = [("tex", "quads"), ("quads", "polys", "tex", "neg", "groups")]     # features of the even / odd seeds


@pytest.mark.parametrize("seed", range(8))
def test_generated_obj_renders_like_the_reference_pipeline(tmp_path, seed):
    """A generated textured OBJ (quads, polygons, random materials, PNG / TGA maps) through BOTH whole pipelines on the CPU: the
    reference's Scene + Bvh + kernels (oracle/_ref, stored as digests) against host loader + host BVH + oracle — primary hits
    and every radiance bit.  (560 further seeds were run once with 0 differences.)"""
    from tests import obj_cases
    obj = obj_cases.write_case(str(tmp_path), obj_cases.random_scene(200 + seed, GENERATED_OBJ[seed % 2]))
    w, h, mb = 96, 54, 5
    cam = hostapi.default_camera(w, h); cam["position"][:3] = (0.2, -3.4, 0.4)
    s = hostapi.HostScene(obj)
    s.add_directional_light((-0.6, -1.5, 3.5), (15, 10, 5)); s.build_bvh()
    env, env_w, env_h = scene_io.load_env()                     # the reference's decoding of its environment map
    s.finalize(env=env, env_width=env_w, env_height=env_h)
    a = s.arrays(); s.close()
    acc, hits, st = Oracle(a).render(cam, w, h, mb)
    ref = reference_record("generated_obj/%d" % seed)
    assert (hits["primitive_id"] != 0xFFFFFFFF).sum() > 100
    assert digest(hits["primitive_id"]) == ref["primitive_id"]
    assert st["n_ext"][: mb + 1].tolist() == ref["n_ext"]
    assert digest(acc[..., :3]) == ref["radiance"]


def test_bvh_builder_on_generated_soups(tmp_path):
    """host/bvh.cpp (SAH buckets, leaf rule, child order; child tasks, chunked passes at the top of the tree) on twelve generated
    triangle soups — uniform, clustered, many identical centroids, a regular grid (ties in every bucket), one axis, coordinates
    with both zeros — against digests of the trees
    the reference's Bvh::BuildCPU built from the same OBJ text (tests/golden/make_obj_fixtures.py)."""
    import json
    from tests import obj_cases
    with open(os.path.join(REPO, "tests", "golden", "obj", "bvh_soups.json")) as f:
        expected = json.load(f)
    for mode, seed, n in obj_cases.SOUP_CASES:
        key = "%s_%d_%d" % (mode, seed, n)
        obj = obj_cases.write_case(str(tmp_path / key), obj_cases.triangle_soup(mode, seed, n))
        assert obj_cases.tree_digest(_scene_arrays_from_obj(obj)) == expected[key], key
    # the tree does not depend on how the build is spread over threads: (threads, nodes above this size run their passes in
    # chunks, children of nodes above this size become tasks)
    saved = {k: os.environ.get(k) for k in ("RT_BVH_THREADS", "RT_BVH_PARALLEL_NODE", "RT_BVH_TASK_NODE")}
    try:
        for threads, par_node, task_node in ((1, 1000, 200), (3, 500, 100), (8, 1000, 200), (5, 64, 16), (8, 1 << 30, 1 << 30)):
            os.environ.update(RT_BVH_THREADS=str(threads), RT_BVH_PARALLEL_NODE=str(par_node), RT_BVH_TASK_NODE=str(task_node))
            for mode, seed, n in obj_cases.SOUP_CASES:
                if n > 3000 and threads not in (3, 8):
                    continue
                key = "%s_%d_%d" % (mode, seed, n)
                assert obj_cases.tree_digest(_scene_arrays_from_obj(str(tmp_path / key / "s.obj"))) == expected[key], (key, threads, par_node, task_node)
    finally:
        for k, v in saved.items():
            os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)


LIVE_OBJ_CASES = [(seed, features) for seed in range(100, 112)
                  for features in (("quads", "polys"), ("quads", "polys", "neg", "groups", "tabs", "crlf", "vcolor", "badmtl", "smooth"))]


def numbers_obj():
    """120 000 numbers in ten notations as vertex coordinates."""
    rng = np.random.default_rng(9)
    vals = np.concatenate([rng.uniform(-3, 3, 60000), rng.normal(0, 100, 30000), 10.0 ** rng.uniform(-6, 4, 30000)])
    rng.shuffle(vals)
    notations = ["%.6f", "%.9f", "%.4e", "%.3f", "%.12g", "%.17g", "%.8f", "%.10e", "%.7f", "%.15f"]
    toks = [notations[i % len(notations)] % v for i, v in enumerate(vals)]
    lines = ["mtllib s.mtl", "vn 0 0 1", "usemtl a"] + ["v %s %s %s" % tuple(toks[3 * i: 3 * i + 3]) for i in range(len(toks) // 3)]
    lines += ["f %d//1 %d//1 %d//1" % (i + 1, i + 2, i + 3) for i in range(0, len(toks) // 3 - 2, 3)]
    return {"s.obj": "\n".join(lines) + "\n", "s.mtl": "newmtl a\nKd 0.5 0.5 0.5\n"}


def test_obj_reader_matches_the_reference_loader_live(tmp_path):
    """Generated scenes (other seeds than tests/golden/obj) and 120 000 numbers in ten notations through host/obj_reader.cpp,
    against digests of what the reference's own loader (oracle/_ref) made of the same files."""
    from tests import hdr_cases, obj_cases
    from tests.ref_cases import scene_arrays_digest
    ref = reference_record("obj_reader_live")
    for k, (seed, features) in enumerate(LIVE_OBJ_CASES):
        obj = obj_cases.write_case(str(tmp_path / ("r%d" % k)), obj_cases.random_scene(seed, features))
        assert scene_arrays_digest(_scene_arrays_from_obj(obj)) == ref["%d_%s" % (seed, "_".join(features))], (seed, features)
    obj = obj_cases.write_case(str(tmp_path / "numbers"), numbers_obj())
    assert scene_arrays_digest(_scene_arrays_from_obj(obj)) == ref["numbers"]
    # environment maps, another seed than the committed digests
    for name, data in hdr_cases.cases(seed=31).items():
        with open(tmp_path / "e.hdr", "wb") as f:
            f.write(data)
        assert hdr_cases.digest(*_load_env(str(tmp_path / "e.hdr"))) == ref["env/" + name], name


TEXTURE_DIR = os.path.join(REPO, "tests", "golden", "textures")


def _load_texture_files(directory, names, tmp_path):
    """{name: (width, height, texels)} through the C++ Scene loader: one material per file, files looked up next to the OBJ."""
    for n in names:
        if not os.path.exists(tmp_path / n):
            os.symlink(os.path.join(directory, n), tmp_path / n)
    with open(tmp_path / "t.mtl", "w") as f:
        for k, n in enumerate(names):
            f.write(f"newmtl m{k}\nKd 0.5 0.5 0.5\nmap_Kd {n}\n")
    with open(tmp_path / "t.obj", "w") as f:
        f.write("mtllib t.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nvn 0 0 1\nvt 0 0\n")
        for k in range(len(names)):
            f.write(f"usemtl m{k}\nf 1/1/1 2/1/1 3/1/1\n")
    s = hostapi.HostScene(str(tmp_path / "t.obj"))
    s.add_directional_light((0, 0, 1), (1, 1, 1))
    s.finalize(env=np.zeros(4, dtype=np.float32), env_width=1, env_height=1)
    a = s.arrays()
    assert len(a["textures"]) == len(names)
    out = {}
    for k, n in enumerate(names):
        t = a["textures"][k]
        count = int(t["width"]) * int(t["height"])
        out[n] = (int(t["width"]), int(t["height"]), a["texels"][int(t["data_start"]): int(t["data_start"]) + count].copy())
    s.close()
    return out


def test_texture_files_decode_like_the_reference(tmp_path):
    """JPEG (baseline / progressive, every chroma layout Pillow writes, greyscale, CMYK, restart intervals) and Adam7 PNG files
    through host/jpeg_decoder.cpp + host/image_loader.cpp against the texel words the reference's own loader (stb_image via
    LoadSTB) produced for the same files (tests/golden/make_texture_fixtures.py).  A JPEG stream does not pin the inverse DCT,
    the chroma filter or the colour conversion — these fixtures do."""
    expected = np.load(os.path.join(TEXTURE_DIR, "expected.npz"))
    names = sorted(k[:-len(":size")] for k in expected.files if k.endswith(":size"))
    assert len(names) >= 50 and all(os.path.exists(os.path.join(TEXTURE_DIR, n)) for n in names)
    got = _load_texture_files(TEXTURE_DIR, names, tmp_path)
    for n in names:
        w, h, texels = got[n]
        assert (w, h) == tuple(expected[n + ":size"]), n
        assert np.array_equal(texels, expected[n + ":texels"]), n
    # the interlaced-PNG writer of the fixture script, against Pillow on the file it can read back
    from PIL import Image
    for n in ("plain_rgb8.png", "a7_rgb8.png", "a7_rgba8.png", "a7_ga8.png", "a7_pal4.png"):
        im = Image.open(os.path.join(TEXTURE_DIR, n))
        assert np.array_equal(_pack_like_stb(im.convert("RGB") if im.mode == "P" else im), expected[n + ":texels"]), n


def textured_obj_images(directory):
    """PNG (RGB, RGBA, grey, grey+alpha, palette with and without tRNS, 16 bit, 1 bit) and TGA (RGB, RLE RGBA, grey) files
    written into `directory`; returns their names."""
    from PIL import Image
    rng = np.random.default_rng(21)

    def rnd(shape, dtype=np.uint8, hi=256):
        return rng.integers(0, hi, size=shape).astype(dtype)
    imgs = {
        "rgb.png": Image.fromarray(rnd((21, 34, 3)), "RGB"),
        "rgba.png": Image.fromarray(rnd((16, 16, 4)), "RGBA"),
        "grey.png": Image.fromarray(rnd((9, 13)), "L"),
        "la.png": Image.fromarray(rnd((8, 8, 2)), "LA"),
        "rgb.tga": Image.fromarray(rnd((12, 10, 3)), "RGB"),
        "rgba_rle.tga": Image.fromarray(np.repeat(rnd((6, 5, 4)), 4, axis=1), "RGBA"),
        "grey.tga": Image.fromarray(rnd((4, 7)), "L"),
    }
    pal = Image.fromarray(rnd((10, 12), hi=16), "P"); pal.putpalette(list(rnd(48)))
    imgs["pal.png"] = pal
    palt = Image.fromarray(rnd((6, 9), hi=4), "P"); palt.putpalette(list(rnd(12)))
    imgs["pal_trns.png"] = palt
    imgs["grey16.png"] = Image.fromarray(rnd((5, 9), np.uint16, 65536))
    imgs["bits1.png"] = Image.fromarray(rnd((11, 19), hi=2) * 255, "L").convert("1")
    for name, im in imgs.items():
        path = os.path.join(str(directory), name)
        if name == "rgba_rle.tga":
            im.save(path, compression="tga_rle")
        elif name == "pal_trns.png":
            im.save(path, transparency=bytes([0, 128, 255, 7]))
        else:
            im.save(path)
    return list(imgs)


def test_image_textures_match_the_reference_loader(tmp_path):
    """The same textured OBJ through host/image_loader.cpp and, stored as digests, through the reference's own Scene (tinyobj +
    LoadSTB, compiled into oracle/_ref): Texture[] records, texel words and packed material words identical
    (scene.cpp:155-186,276-300); then freshly generated JPEG / Adam7 files and the reference's assets/checker3.jpg."""
    ref = reference_record("image_textures")
    obj = _textured_obj(tmp_path, textured_obj_images(tmp_path))
    s = hostapi.HostScene(obj)
    s.add_directional_light((-0.6, -1.5, 3.5), (15, 10, 5))
    s.build_bvh()
    s.finalize(env=np.zeros(4, dtype=np.float32), env_width=1, env_height=1)
    a = s.arrays()
    assert len(a["textures"]) == ref["textures"]
    for f in ("width", "height", "data_start"):                   # the record's padding word is uninitialised in the reference
        assert digest(a["textures"][f]) == ref[f], f
    assert digest(a["texels"]) == ref["texels"]
    assert digest(a["materials"]) == ref["materials"]
    assert digest(a["triangles"]["mtlIndex"]) == ref["mtlIndex"]
    for v in ("v1", "v2", "v3"):
        assert digest(a["triangles"][v]["texcoord"][:, :2]) == ref[v + ".texcoord"], v
    s.close()
    # freshly generated JPEG / Adam7 files (another seed than the committed fixtures)
    from tests.golden import make_texture_fixtures as mk
    fresh = tmp_path / "fresh"
    names = mk.make_files(str(fresh), np.random.default_rng(77))
    assert sorted(names) == sorted(ref["fresh"])
    work = tmp_path / "work"; work.mkdir()
    got = _load_texture_files(str(fresh), names, work)
    for n in names:
        w, h, texels = got[n]
        assert [w, h, digest(texels)] == ref["fresh"][n], n
    # the JPEG the reference ships with its assets
    work = tmp_path / "assets"; work.mkdir()
    for n, (w, h, texels) in _load_texture_files(REF_GOLDEN, sorted(ref["assets"]), work).items():
        assert [w, h, digest(texels)] == ref["assets"][n], n


@pytest.mark.gpu
def test_textured_obj_renders_like_the_oracle(tmp_path):
    """OBJ with image textures -> C++ Scene (image_loader.cpp) -> Render(kCUDA) -> the texture sampling path of the kernels
    (material.h:251-264,319-369), against the oracle on the arrays the loader produced."""
    from PIL import Image
    rng = np.random.default_rng(8)
    names = ["a.png", "b.tga", "c.png", "d.png", "e.tga", "f.png"]
    for n in names:
        Image.fromarray(rng.integers(0, 256, size=(16, 16, 4 if n != "c.png" else 3)).astype(np.uint8)).save(str(tmp_path / n))
    env_path, _ = make_env(tmp_path, w=64, h=32)
    w, h, mb = 160, 90, 4
    s = hostapi.HostScene(_textured_obj(tmp_path, names))
    s.add_directional_light((-0.3, -0.4, 1.0), (8, 8, 8))
    r = hostapi.HostRender(s, w, h, env_path)
    r.set_max_bounces(mb)
    cam = hostapi.default_camera(w, h); cam["position"][:3] = (4.0, -2.5, 1.6)
    r.set_camera(cam)
    a = s.arrays(); a["nodes"] = r.nodes()
    assert len(a["textures"]) == 6
    o = Oracle(a)
    r.render_frame()
    acc, _, ost = o.render(cam, w, h, mb)
    assert ost["n_ext"][1] > 500 and ost["n_shadow"][0] > 300           # the quads are in view and lit
    expect = acc[..., :3] / (acc[..., :3] + np.float32(1.0))
    assert np.array_equal(bits(r.image()[..., :3]), bits(expect))
    r.close(); s.close()


@pytest.mark.parametrize("name", ["CornellBox", "ShaderBalls", "CornellBox_Dragon"])
def test_loader_and_builder_reproduce_reference_dumps(tmp_path, name):
    """Same OBJ/MTL/HDR in -> the arrays the reference's own Scene + Bvh::BuildCPU + LoadHDR produced (stored per field as
    digests).  CornellBox is the reference's whole OBJ; of the two large ones, runs of 64 consecutive faces, one in every 128, with
    the lines they use are kept (tests/ref_cases.py: obj_face_subset).  The environment map is read from every 50th scanline of the reference's file and
    compared with those rows of its decoding."""
    from tests.ref_cases import ENV_ROW_STEP, loader_digests, write_env_rows, write_loader_input
    s = hostapi.HostScene(write_loader_input(name, tmp_path))
    s.add_directional_light((-0.6, -1.5, 3.5), (15, 10, 5))      # main.cpp:58
    s.build_bvh()
    s.finalize(env_path=write_env_rows(tmp_path))
    a = s.arrays()
    got, ref = loader_digests(a), reference_record("loader/" + name)
    assert [k for k in ref if got[k] != ref[k]] == [], (got["counts"], ref["counts"])
    env, env_w, env_h = scene_io.load_env()
    rows = env.reshape(env_h, env_w, 4)[::ENV_ROW_STEP]
    assert (int(a["env_width"]), int(a["env_height"])) == (rows.shape[1], rows.shape[0])
    assert np.array_equal(bits(a["env"]), bits(rows.reshape(-1)))
    s.close()


def test_standalone_bvh_build_on_fixture_triangles():
    g = scene("ShaderBalls")
    rng = np.random.default_rng(0)
    shuffled = g["triangles"][rng.permutation(len(g["triangles"]))][:5000]
    tris, nodes, depth = hostapi.build_bvh(shuffled)
    assert len(tris) == 5000 and depth <= 64
    assert sorted(map(bytes, tris)) == sorted(map(bytes, shuffled))       # a permutation of the input
    count = nodes["num_primitives_axis"] >> 16
    assert count[count > 0].sum() == 5000


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", ["frame", "fused", "stepwise"])
def test_render_kcuda_over_several_devices_matches_oracle(tmp_path, schedule):
    """Render(kCUDA, devices): ONE CUDAPathTraceIntegrator over several GPUs behind the unchanged Integrator interface (the
    devices of the box, or device 0 listed twice when it has one) — Integrate() x3 in every schedule, resolved image against
    the oracle.  "frame" is the deferred schedule: the virtuals only check their order and AdvanceSampleCount submits the frame."""
    from raytracing_b200 import capi
    w, h, mb = 180, 101, 5
    env_path, _ = make_env(tmp_path, w=64, h=32)
    s = hostapi.HostScene(PROC_OBJ)
    s.add_directional_light((-0.6, -1.5, 3.5), (15, 10, 5))
    n_dev = capi.device_count()
    r = hostapi.HostRender(s, w, h, env_path, devices=list(range(n_dev)) if n_dev >= 2 else [0, 0], schedule=schedule)
    r.set_max_bounces(mb)
    a = s.arrays(); a["nodes"] = r.nodes()
    o = Oracle(a)
    cam = hostapi.default_camera(w, h)
    acc = np.zeros((h, w, 4), dtype="<f4")
    for sample in range(3):
        r.render_frame()
        acc, _, _ = o.render(cam, w, h, mb, sample_idx=sample, radiance=acc)
        hdr = acc[..., :3] / np.float32(sample + 1)
        assert np.array_equal(bits(r.image()[..., :3]), bits(hdr / (hdr + np.float32(1.0)))), (schedule, sample)
    r.close(); s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("stepwise", [False, True], ids=["frame", "stepwise"])
def test_render_kcuda_backend_matches_oracle(tmp_path, stepwise):
    """The whole C++ host path — Scene(OBJ) -> Render(kCUDA) -> Bvh::BuildCPU -> Finalize -> CUDAPathTraceIntegrator
    -> UploadGPUData -> RenderFrame() x2 (Integrator::Integrate schedule) — against the oracle on the same arrays."""
    w, h, mb = 200, 120, 6
    env_path, _ = make_env(tmp_path, w=64, h=32)
    s = hostapi.HostScene(PROC_OBJ)
    s.add_directional_light((-0.6, -1.5, 3.5), (15, 10, 5))
    s.add_point_light((0.5, 0.2, 2.0), (4, 4, 6))
    r = hostapi.HostRender(s, w, h, env_path, stepwise=stepwise)
    r.set_max_bounces(mb)
    a = s.arrays()                       # after Render built the BVH (reordering the triangles) and finalized the scene
    a["nodes"] = r.nodes()               # Render owns the acceleration structure
    o = Oracle(a)
    cam = hostapi.default_camera(w, h)
    acc = np.zeros((h, w, 4), dtype="<f4")
    for sample in range(2):
        r.render_frame()
        acc, _, _ = o.render(cam, w, h, mb, sample_idx=sample, radiance=acc)
        hdr = acc[..., :3] / np.float32(sample + 1)              # resolve_radiance.cl:80-84
        expect = hdr / (hdr + np.float32(1.0))
        img = r.image()
        assert np.array_equal(bits(img[..., :3]), bits(expect)), sample
        assert (img[..., 3] == 1.0).all()
    # option setters keep the reference behaviour: kBlueNoise without its tables fails loudly; with them the next frame
    # restarts the accumulation with the other sampler; white furnace re-renders from scratch
    with pytest.raises(hostapi.HostError):
        r.set_blue_noise(True)
    tables = synthetic_sampler_tables()
    r.set_blue_noise_tables(*tables)
    r.set_blue_noise(True)
    r.render_frame()
    try:
        o.set_sampler_tables(tables)
        bn, _, _ = o.render(cam, w, h, mb, sample_idx=0)
    finally:
        o.set_sampler_tables(None)
    assert np.array_equal(bits(r.image()[..., :3]), bits(bn[..., :3] / (bn[..., :3] + np.float32(1.0))))
    r.set_blue_noise(False)
    r.enable_white_furnace(True)
    r.render_frame()
    wf, _, _ = o.render(cam, w, h, mb, sample_idx=0, white_furnace=True)
    expect = wf[..., :3] / (wf[..., :3] + np.float32(1.0))
    assert np.array_equal(bits(r.image()[..., :3]), bits(expect))
    r.close(); s.close()
