"""
CPU tests (-m "not gpu"): the oracle restatement against what the reference's own kernels (oracle/_ref) computed on
configurations other than the committed golden ones (different resolution / bounce count / sample index / options),
stored by tests/golden/make_ref_fixtures.py as per-bounce counters and digests of the outputs.  Bar: bit-exact.
"""
import json
import os

import numpy as np
import pytest

from oracle.orcbind import Oracle
from raytracing_b200.camera import default_camera
from tests.helpers import bits, digest, fuzz_configs, scene, synthetic_sampler_tables
from tests.ref_cases import (AOV_CAMERAS, BIT_EXACT, BLUE_NOISE, DEGENERATE, LIBM, LIGHTS_LENS, OUT, STATS, frame_key, libm_pixels,
                             lights_lens_camera)

with open(os.path.join(OUT, "expected.json")) as _f:
    REF = json.load(_f)


def check_sample(ref, mb, acc, hits, st, keys=STATS, sample=0):
    for k in keys:
        assert st[k][: mb + 1].tolist() == ref[k], (k, sample)
    if hits is not None:
        assert digest(hits["primitive_id"]) == ref["primitive_id"], ("primary hits", sample)
    assert digest(acc[..., :3]) == ref["radiance"], ("radiance", sample)


def progressive(o, ref, cam, w, h, mb, wf=False):
    acc = np.zeros((h, w, 4), dtype="<f4")
    for sample, rs in enumerate(ref):           # progressive accumulation: sample_idx 0, 1, ...
        acc, hits, st = o.render(cam, w, h, mb, sample_idx=sample, white_furnace=wf, radiance=acc)
        check_sample(rs, mb, acc, hits, st, sample=sample)
    return st


@pytest.mark.parametrize("name,w,h,mb,wf", BIT_EXACT)
def test_oracle_bit_exact_vs_reference_kernels(name, w, h, mb, wf):
    progressive(Oracle(scene(name)), REF["bit_exact/" + frame_key(name, w, h, mb, wf)], default_camera(w, h), w, h, mb, wf)


@pytest.mark.parametrize("name", ["CornellBox", "ShaderBalls"])
def test_aov_denoiser_resolve_restatements_vs_reference_kernels(name):
    """orc_aovs / orc_temporal_accumulation / orc_resolve against aov.cl, denoiser.cl, resolve_radiance.cl (3 frames, moving camera)."""
    sc = scene(name); w, h, mb = 128, 72, 3
    o = Oracle(sc)
    cams = [default_camera(w, h, **kw) for kw in AOV_CAMERAS]
    prev = np.zeros((), dtype=cams[0].dtype)
    prev_rad = np.zeros((h, w, 4), "<f4"); prev_depth = np.zeros((h, w), "<f4")
    for f, (cam, ref) in enumerate(zip(cams, REF["aov/" + name])):
        rad, _, _ = o.render(cam, w, h, mb, sample_idx=f)
        al, de, no, ve = o.aovs(cam, prev, w, h, sample_idx=f)
        assert digest(al[..., :3]) == ref["albedo"] and digest(de) == ref["depth"]
        assert digest(no[..., :3]) == ref["normal"] and digest(ve) == ref["velocity"]
        den = o.temporal_accumulation(rad, prev_rad, de, prev_depth, ve)
        assert digest(den[..., :3]) == ref["radiance"]
        assert digest(o.resolve(0, den, al, de, no, ve, f + 1, denoiser=True)) == ref["resolved"]
        prev_rad, prev_depth, prev = den, de, cam


def test_textured_materials_bit_exact_vs_reference_kernels():
    """ApplyTextures / SampleTexture (material.h:251-264,319-369) on every texture slot, wrapped coordinates included."""
    from tests.scenes_extra import textured_cornell
    sc = textured_cornell()
    w, h, mb = 96, 64, 4
    cam = default_camera(w, h)
    rad, hits, st = Oracle(sc).render(cam, w, h, mb)
    check_sample(REF["textured"], mb, rad, hits, st)
    # the textured image must differ from the untextured one (the textures are really used)
    plain, _, _ = Oracle(scene("CornellBox")).render(cam, w, h, mb)
    assert not np.array_equal(bits(plain), bits(rad))


@pytest.mark.parametrize("name,w,h,mb,wf", BLUE_NOISE)
def test_blue_noise_sampler_bit_exact_vs_reference_kernels(name, w, h, mb, wf):
    """SamplerType::kBlueNoise (sampling.h:40-61): the restatement against hit_surface.cl built with -DBLUE_NOISE_SAMPLER, both
    reading the same seeded stand-in tables (the reference's own tables are reference data), three progressive samples."""
    o = Oracle(scene(name))
    cam = default_camera(w, h)
    tables = synthetic_sampler_tables()
    try:
        o.set_sampler_tables(tables)
        progressive(o, REF["blue_noise/" + frame_key(name, w, h, mb, wf)], cam, w, h, mb, wf)
        # and the sampler did change the image
        o.set_sampler_tables(None)
        plain, _, _ = o.render(cam, w, h, mb, sample_idx=0, white_furnace=wf)
        first, _, _ = (o.set_sampler_tables(tables), o.render(cam, w, h, mb, sample_idx=0, white_furnace=wf))[1]
        assert not np.array_equal(bits(plain), bits(first))
    finally:
        o.set_sampler_tables(None)


@pytest.mark.parametrize("name,w,h,mb", LIGHTS_LENS)
def test_point_lights_and_thin_lens_bit_exact_vs_reference_kernels(name, w, h, mb):
    """Five analytic lights (point + directional, light.h:30-65) and a thin-lens camera (aperture > 0: the hexagonal
    aperture sampling of raygeneration.cl:40-49,108-124), moved off the default pose."""
    from tests.scenes_extra import many_lights_scene
    st = progressive(Oracle(many_lights_scene(name)), REF["lights_lens/" + name], lights_lens_camera(w, h), w, h, mb)
    assert st["n_shadow"][:mb].min() > 0 and st["n_unoccluded"][:mb].min() > 0


@pytest.mark.parametrize("case", list(DEGENERATE))
def test_degenerate_frames_bit_exact_vs_reference_kernels(case):
    """max_bounces = 0 (one extension pass, one shadow pass); a camera that only sees the sky (every queue after bounce 0
    is empty); a camera placed inside a ShaderBall (rays start inside closed geometry: back faces are culled)."""
    name, w, h, mb, kw = DEGENERATE[case]
    st = progressive(Oracle(scene(name)), REF["degenerate/" + case], default_camera(w, h, **kw), w, h, mb)
    if case == "all_miss":
        assert st["n_hit"][0] == 0 and st["n_ext"][1] == 0


@pytest.mark.parametrize("cfg", fuzz_configs(), ids=lambda c: f"{c[0]}_{c[1]}x{c[2]}_b{c[3]}")
def test_fuzzed_frames_bit_exact_vs_reference_kernels(cfg):
    """Seeded random scenes / sizes / bounce counts / camera poses and lenses, two progressive samples each."""
    name, w, h, mb, kw, wf = cfg
    ref = REF["fuzz/%d" % fuzz_configs().index(cfg)]
    progressive(Oracle(scene(name)), ref, default_camera(w, h, **kw), w, h, mb, wf)


@pytest.mark.parametrize("name,w,h,mb,limit", LIBM)
def test_math_library_sensitivity_is_small(name, w, h, mb, limit):
    """The OpenCL driver's libm is unpinned (SURVEY 8c).  The reference kernels with glibc's libm in place of include/rt_math.h
    (a seeded sample of their pixels is stored) must leave all but a small fraction of pixels within 1e-4 relative of the
    oracle, which is bit-identical to the reference kernels with include/rt_math.h — on all three shipped scenes (the mirror /
    metal paths of the Dragon scene at 16 bounces are the most sensitive).  include/rt_math.h itself is pinned against
    double-precision libm in tests/test_rt_math.py."""
    rad, _, _ = Oracle(scene(name)).render(default_camera(w, h), w, h, mb)
    assert digest(rad[..., :3]) == REF["libm/" + name]["radiance"]
    a = rad[..., :3].reshape(-1, 3)[libm_pixels(w, h)].astype(np.float64)
    b = np.load(os.path.join(OUT, "libm_samples.npz"))[name].astype(np.float64)
    rel = np.abs(a - b) / np.maximum(np.abs(a), 1e-6)
    frac_bad = (rel.max(axis=-1) > 1e-4).mean()
    assert frac_bad < limit, frac_bad
