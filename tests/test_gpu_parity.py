"""
GPU parity tests (-m gpu): the CUDA path, called through the C ABI (include/rt_b200.h),
against the CPU oracle on the same seeded inputs and against the golden vectors produced
by the reference's own kernels (tests/golden/).

Bar (BASELINE.json north_star: "bit-exact primary-hit triangle indices and per-pixel
radiance within 1e-4 relative"): this implementation is held to the stricter BIT-EXACT bar
for everything — hit indices, barycentrics, per-bounce ray counters and every radiance
float — because oracle and kernels share one arithmetic policy (DESIGN.md).
"""
import os

import numpy as np
import pytest

from oracle.orcbind import Oracle
from raytracing_b200 import capi
from raytracing_b200.camera import default_camera
from tests.helpers import bits, fuzz_configs, golden_files, load_golden, scene, synthetic_sampler_tables

pytestmark = pytest.mark.gpu

INVALID = 0xFFFFFFFF


def make_ctx(name, w, h, **kw):
    ctx = capi.Context(w, h, **kw)
    ctx.upload_scene(scene(name))
    ctx.set_camera(default_camera(w, h))
    return ctx


def check_stats(st, ost, mb):
    for k in ("n_ext", "n_miss", "n_shadow", "n_cont", "n_unoccluded", "n_emissive_hits"):
        assert np.array_equal(st[k][: mb + 1], ost[k][: mb + 1]), k


@pytest.mark.parametrize("path", golden_files(), ids=lambda p: p.split("golden_")[-1].replace(".npz.xz", ""))
@pytest.mark.parametrize("fused", [False, True], ids=["stepwise", "fused"])
def test_matches_reference_golden(path, fused):
    """CUDA vs outputs of the reference's own kernels (committed fixtures)."""
    g = load_golden(path)
    w, h, mb = int(g["width"]), int(g["height"]), int(g["max_bounces"])
    ctx = capi.Context(w, h)
    ctx.upload_scene(scene(g["scene_name"]))
    ctx.set_camera(g["camera"])
    ctx.set_option(capi.OPT_WHITE_FURNACE, int(g["white_furnace"]))
    ctx.reset()
    for _ in range(int(g["sample_count"]) - 1):               # progressive fixtures: the earlier samples
        ctx.integrate(mb) if fused else ctx.integrate_stepwise(mb)
    if fused:
        ctx.integrate(mb)
    else:
        ctx.generate_rays()
        ctx.intersect(0)
        hits, pix = ctx.read_hits(0)
        prim = np.full(w * h, 0xFFFFFFFE, dtype=np.uint32)
        prim[pix] = hits["primitive_id"]
        assert np.array_equal(prim, g["primitive_id"])          # bit-exact primary-hit triangle indices
        if "hit_bc" in g:
            hit = g["primitive_id"] != INVALID
            bc = np.zeros((w * h, 2), dtype=np.float32); bc[pix] = hits["bc"]
            t = np.zeros(w * h, dtype=np.float32); t[pix] = hits["t"]
            assert np.array_equal(bits(bc[hit]), bits(g["hit_bc"][hit]))
            assert np.array_equal(bits(t[hit]), bits(g["hit_t"][hit]))
            rays, rpix = ctx.read_rays(0)
            o = np.zeros((w * h, 4), dtype=np.float32); o[rpix] = rays["origin"]
            d = np.zeros((w * h, 4), dtype=np.float32); d[rpix] = rays["direction"]
            assert np.array_equal(bits(o), bits(g["ray_origin"]))
            assert np.array_equal(bits(d), bits(g["ray_direction"]))
        ctx.integrate_stepwise(mb)
    rad = ctx.read_radiance()
    st = ctx.frame_stats()
    for k in ("n_ext", "n_miss", "n_shadow", "n_cont", "n_unoccluded"):
        assert np.array_equal(st[k][: mb + 1], g[k]), k
    assert np.array_equal(bits(rad[..., :3]), bits(g["radiance_rgb"]))
    assert ctx.sample_count() == int(g["sample_count"])
    if "resolved" in g:
        res = ctx.resolve()
        assert np.array_equal(bits(res), bits(g["resolved"]))
    ctx.destroy()


@pytest.mark.parametrize("name,w,h,mb", [
    ("CornellBox", 256, 256, 2),          # BASELINE config C1
    ("CornellBox", 333, 127, 8),          # ragged size: last warp / last block partially filled
    ("ShaderBalls", 480, 270, 8),
    ("CornellBox_Dragon", 384, 216, 16),
])
@pytest.mark.parametrize("traversal", [0, 1], ids=["literal", "fast"])
def test_fused_and_stepwise_match_oracle(name, w, h, mb, traversal):
    """CUDA (both schedules, both traversal kernels) vs the CPU oracle, live, two accumulated samples."""
    sc = scene(name)
    cam = default_camera(w, h)
    o = Oracle(sc)
    oacc = np.zeros((h, w, 4), dtype="<f4")
    ctxs = {}
    for mode in ("fused", "stepwise"):
        c = make_ctx(name, w, h)
        c.set_option(capi.OPT_TRAVERSAL, traversal)
        c.reset()
        ctxs[mode] = c
    for sample in range(2):
        oacc, ohits, ost = o.render(cam, w, h, mb, sample_idx=sample, radiance=oacc)
        ctxs["fused"].integrate(mb)
        ctxs["stepwise"].integrate_stepwise(mb)
        for mode, c in ctxs.items():
            check_stats(c.frame_stats(), ost, mb)
            assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(oacc[..., :3])), (mode, sample)
    for c in ctxs.values():
        c.destroy()


def test_traversal_work_counters_match_oracle():
    """RT_OPT_COUNT_TRAVERSAL: nodes visited / triangles tested in reference order (the algorithmic-bytes inputs)."""
    name, w, h, mb = "ShaderBalls", 320, 180, 4
    cam = default_camera(w, h)
    _, _, ost = Oracle(scene(name)).render(cam, w, h, mb)
    c = make_ctx(name, w, h)
    c.set_option(capi.OPT_COUNT_TRAVERSAL, 1)
    c.reset(); c.integrate(mb)
    st = c.frame_stats()
    for k in ("nodes_ext", "tris_ext", "nodes_shadow", "tris_shadow"):
        assert np.array_equal(st[k][: mb + 1], ost[k][: mb + 1]), k
    c.destroy()


def test_white_furnace_and_empty_tail():
    """White furnace (energy aid, SURVEY 4) + more bounces than any path survives (empty queues must be harmless)."""
    name, w, h, mb = "CornellBox", 128, 96, 40
    cam = default_camera(w, h)
    orad, _, ost = Oracle(scene(name)).render(cam, w, h, mb, white_furnace=True)
    c = make_ctx(name, w, h)
    c.set_option(capi.OPT_WHITE_FURNACE, 1)
    c.reset(); c.integrate(mb)
    rad = c.read_radiance()
    assert np.array_equal(bits(rad[..., :3]), bits(orad[..., :3]))
    assert np.isfinite(rad).all()
    # pixels whose paths never picked up the analytic light see only the 0.5-grey sky: never more than 0.5 (+rounding)
    st = c.frame_stats()
    assert st["n_ext"][mb] == 0 or st["n_ext"][mb] < st["n_ext"][0]
    c.destroy()


@pytest.mark.parametrize("world", [2, 3])
def test_scanline_partition_reassembles_bit_exact(world):
    """Multi-GPU partition on one device: each rank renders rows y % world == rank; the union equals the full frame."""
    name, w, h, mb = "ShaderBalls", 200, 101, 5
    full = make_ctx(name, w, h)
    full.reset(); full.integrate(mb)
    ref = full.read_radiance()
    out = np.zeros_like(ref)
    for rank in range(world):
        c = make_ctx(name, w, h, rank=rank, world=world)
        c.reset(); c.integrate(mb)
        c.read_radiance(out)
        c.destroy()
    assert np.array_equal(bits(out), bits(ref))
    full.destroy()


def test_gathered_frame_resolves_like_a_single_gpu_frame():
    """rt_resolve_gathered on the gathering rank: three partitions rendered by three contexts, their radiance slabs laid
    out the way the NCCL gather delivers them, resolved through the scanline map — equal to rt_resolve of one context
    that rendered the whole image.  Height 101 is not a multiple of 3 (ragged last rows, padded slabs)."""
    import torch
    from raytracing_b200.distributed import RadianceGather, local_rows
    w, h, mb, world = 160, 101, 4, 3
    whole = make_ctx("CornellBox", w, h); whole.reset()
    parts = [capi.Context(w, h, rank=r, world=world) for r in range(world)]
    for c in parts:
        c.upload_scene(scene("CornellBox")); c.set_camera(default_camera(w, h)); c.reset()
    for _ in range(2):
        whole.integrate(mb)
        for c in parts:
            c.integrate(mb)
    g = RadianceGather(w, h, 0, world, torch.device("cuda", 0))
    for r, c in enumerate(parts):
        c.sync()
        ptr, nbytes = c.radiance_device_ptr()
        n = c.local_pixel_count()
        assert n == local_rows(h, r, world) * w and nbytes >= n * 16

        class _Slab:
            __cuda_array_interface__ = {"shape": (n, 4), "typestr": "<f4", "data": (ptr, False), "version": 3, "strides": None}
        g.recv_all[r, :n].copy_(torch.as_tensor(_Slab(), device="cuda"))
    torch.cuda.synchronize()
    want = whole.resolve()
    got = parts[0].resolve_gathered(g.recv_ptr, g.recv_stride_bytes)
    assert np.array_equal(bits(got), bits(want))
    import torch as _t
    host = _t.zeros((h, w, 4), dtype=_t.float32).pin_memory().numpy()
    parts[0].resolve_gathered(g.recv_ptr, g.recv_stride_bytes, out=host, wait=False); parts[0].resolve_wait()
    assert np.array_equal(bits(host), bits(want))
    with pytest.raises(capi.RtError):
        parts[0].resolve_gathered(g.recv_ptr, 64)          # stride cannot hold a slab
    for c in parts + [whole]:
        c.destroy()


@pytest.mark.parametrize("name,w,h,mb,row_first,row_step", [
    ("CornellBox", 1920, 1080, 8, 5, 17),              # BASELINE C2: 64 oracle rows
    ("ShaderBalls", 1920, 1080, 8, 3, 23),             # C3: 47 oracle rows
    ("CornellBox_Dragon", 3840, 2160, 16, 11, 97),     # C4: 23 oracle rows of the 4K frame, 16 bounces
])
def test_full_size_properties(name, w, h, mb, row_first, row_step):
    """The benchmarked configurations AT THE BENCHMARKED SIZE: the three schedules (per-phase kernels, one-kernel frame,
    stepwise) agree bit for bit on the whole frame; live-ray counters are monotone and consistent; a band of rows spread over
    the frame equals the oracle."""
    a = make_ctx(name, w, h); a.set_option(capi.OPT_FRAME_KERNEL, 0)
    f = make_ctx(name, w, h); f.set_option(capi.OPT_FRAME_KERNEL, 1)
    b = make_ctx(name, w, h)
    for c in (a, f, b):
        c.reset()
    a.integrate(mb); f.integrate(mb); b.integrate_stepwise(mb)
    ra, rf, rb = a.read_radiance(), f.read_radiance(), b.read_radiance()
    assert np.array_equal(bits(ra), bits(rb))
    assert np.array_equal(bits(ra), bits(rf))
    st = a.frame_stats()
    for k in ("n_ext", "n_miss", "n_shadow", "n_cont", "n_unoccluded", "n_emissive_hits"):
        assert np.array_equal(st[k][: mb + 1], f.frame_stats()[k][: mb + 1]), k
    n_ext = st["n_ext"][: mb + 1]
    assert n_ext[0] == w * h and (np.diff(n_ext.astype(np.int64)) <= 0).all()
    assert np.array_equal(st["n_cont"][:mb], n_ext[1:])
    assert (st["n_shadow"][: mb + 1] <= n_ext - st["n_miss"][: mb + 1]).all()
    assert (st["n_unoccluded"][: mb + 1] <= st["n_shadow"][: mb + 1]).all()
    orad, _, _ = Oracle(scene(name)).render(default_camera(w, h), w, h, mb, row_first=row_first, row_step=row_step)
    rows = np.arange(row_first, h, row_step)
    assert np.array_equal(bits(ra[rows][..., :3]), bits(orad[rows][..., :3]))
    for c in (a, f, b):
        c.destroy()


def test_full_size_synthetic_10m_triangles():
    """BASELINE C5 at full size: 183 copies of ShaderBalls + ground = 10 026 572 triangles, 1920x1080, 8 bounces (scene and host BVH
    build included: ~30 s on the GPU box, profiles/r02_full_size_parity.txt).  Per-phase kernels == one-kernel frame on the whole frame, a band of 31 rows
    equals the oracle, and more than 90 % of the primary rays hit geometry."""
    from raytracing_b200 import scene_io, synthetic
    w, h, mb = 1920, 1080, 8
    sc = synthetic.bistro_scale_scene(scene_io.load_scene("ShaderBalls"), 183, w, h)
    cam = sc["camera_pose"]
    imgs = []
    for fk in (0, 1):
        c = capi.Context(w, h); c.set_option(capi.OPT_FRAME_KERNEL, fk)
        c.upload_scene(sc); c.set_camera(cam); c.reset(); c.integrate(mb)
        imgs.append(c.read_radiance()); st = c.frame_stats(); c.destroy()
    assert np.array_equal(bits(imgs[0]), bits(imgs[1]))
    assert 1.0 - st["n_miss"][0] / st["n_ext"][0] > 0.9
    orad, _, _ = Oracle(sc).render(cam, w, h, mb, row_first=7, row_step=35)
    rows = np.arange(7, h, 35)
    assert np.array_equal(bits(imgs[0][rows][..., :3]), bits(orad[rows][..., :3]))


def test_synthetic_field_matches_oracle():
    """BASELINE config C5 at reduced scale: 4 copies of ShaderBalls (219 160 triangles, BVH built by the host builder),
    raised camera; CUDA == oracle bit for bit."""
    from raytracing_b200 import scene_io, synthetic
    w, h, mb = 320, 180, 8
    sc = synthetic.bistro_scale_scene(scene_io.load_scene("ShaderBalls"), 4, w, h)
    cam = sc["camera_pose"]
    orad, ohits, ost = Oracle(sc).render(cam, w, h, mb)
    c = capi.Context(w, h)
    c.upload_scene(sc); c.set_camera(cam); c.reset()
    c.generate_rays(); c.intersect(0)
    hits, pix = c.read_hits(0)
    prim = np.zeros(w * h, dtype=np.uint32); prim[pix] = hits["primitive_id"]
    assert np.array_equal(prim, ohits["primitive_id"])
    c.reset(); c.integrate(mb)
    check_stats(c.frame_stats(), ost, mb)
    assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(orad[..., :3]))
    c.destroy()


def test_aovs_denoiser_and_views_match_oracle():
    """SURVEY 8f rows: GenerateAOV (aov.cl), TemporalAccumulation (denoiser.cl), ResolveRadiance views — three frames with
    a moving camera and the denoiser on (sample index keeps counting, radiance is re-initialised every frame)."""
    name, w, h, mb = "ShaderBalls", 192, 108, 3
    sc = scene(name)
    o = Oracle(sc)
    c = capi.Context(w, h)
    c.upload_scene(sc)
    c.set_option(capi.OPT_DENOISER, 1)
    cams = [default_camera(w, h), default_camera(w, h, position=(0.05, -1.02, 1.01)), default_camera(w, h, position=(0.05, -1.02, 1.01))]
    prev_cam = np.zeros((), dtype=cams[0].dtype)
    prev_rad = np.zeros((h, w, 4), "<f4"); prev_depth = np.zeros((h, w), "<f4")
    for f, cam in enumerate(cams):
        c.set_camera(cam)
        # Integrator::Integrate with the denoiser enabled (integrator.cpp:27-59)
        c.reset(); c.generate_rays()
        for b in range(mb + 1):
            c.intersect(b)
            if b == 0:
                c.compute_aovs()
            c.shade_miss(b); c.shade_hits(b); c.intersect_shadow(); c.accumulate_direct()
        c.advance_sample_count(); c.denoise(); c.copy_history()
        img = c.resolve()
        rad, _, _ = o.render(cam, w, h, mb, sample_idx=f)
        al, de, no, ve = o.aovs(cam, prev_cam, w, h, sample_idx=f)
        gal, gde, gno, gve = c.read_aovs()
        assert np.array_equal(bits(gal[..., :3]), bits(al[..., :3])) and np.array_equal(bits(gde), bits(de))
        assert np.array_equal(bits(gno[..., :3]), bits(no[..., :3])) and np.array_equal(bits(gve), bits(ve))
        den = o.temporal_accumulation(rad, prev_rad, de, prev_depth, ve)
        assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(den[..., :3])), f
        assert np.array_equal(bits(img), bits(o.resolve(0, den, al, de, no, ve, f + 1, denoiser=True))), f
        prev_rad, prev_depth, prev_cam = den, de, cam
    for view in (1, 2, 3, 4):
        c.set_option(capi.OPT_AOV, view)
        assert np.array_equal(bits(c.resolve()), bits(o.resolve(view, den, al, de, no, ve, 3, denoiser=True))), view
    c.destroy()
    # fused schedule + AOV view without the denoiser
    c = make_ctx(name, w, h)
    c.set_option(capi.OPT_AOV, 3)
    c.reset(); c.integrate(mb)
    al, de, no, ve = o.aovs(default_camera(w, h), np.zeros((), dtype=cams[0].dtype), w, h)
    assert np.array_equal(bits(c.resolve()[..., :3]), bits(no[..., :3] * np.float32(0.5) + np.float32(0.5)))
    c.destroy()


def test_resolve_async_matches_blocking_resolve():
    name, w, h, mb = "CornellBox", 160, 90, 3
    c = make_ctx(name, w, h)
    c.reset(); c.integrate(mb)
    ref = c.resolve()
    bufs = [np.zeros((h, w, 4), "<f4") for _ in range(3)]
    for b in bufs:                      # three calls: both resolve buffers get re-used
        c.resolve_async(b)
    c.resolve_wait()
    for b in bufs:
        assert np.array_equal(bits(b), bits(ref))
    c.destroy()


def test_textured_materials_match_oracle():
    """Texture sampling path of the shader (per-hit unpack instead of the precomputed material record)."""
    from tests.scenes_extra import textured_cornell
    sc = textured_cornell()
    w, h, mb = 200, 150, 5
    cam = default_camera(w, h)
    orad, _, ost = Oracle(sc).render(cam, w, h, mb)
    for stepwise in (False, True):
        c = capi.Context(w, h); c.upload_scene(sc); c.set_camera(cam); c.reset()
        c.integrate_stepwise(mb) if stepwise else c.integrate(mb)
        check_stats(c.frame_stats(), ost, mb)
        assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(orad[..., :3]))
        c.destroy()


@pytest.mark.parametrize("tables", ["synthetic"])     # seeded stand-ins: the reference's own tables are reference data
@pytest.mark.parametrize("name,w,h,mb,wf", [
    ("CornellBox", 160, 136, 3, False),      # > 128 x 128: all tile pixels, incl. those whose ranking index runs past the table
    ("ShaderBalls", 272, 144, 8, False),
    ("CornellBox", 64, 64, 5, True),
])
def test_blue_noise_sampler_matches_oracle(name, w, h, mb, wf, tables):
    """SetSamplerType(kBlueNoise): all three schedules vs the oracle (itself pinned to hit_surface.cl -DBLUE_NOISE_SAMPLER
    in tests/test_oracle_vs_ref.py), three progressive samples, then back to kRandom."""
    t = synthetic_sampler_tables()
    sc = scene(name); cam = default_camera(w, h)
    o = Oracle(sc)
    ctxs = {}
    for mode in ("fused", "stepwise"):
        c = make_ctx(name, w, h)
        c.set_option(capi.OPT_WHITE_FURNACE, int(wf))
        c.upload_sampler_tables(*t)
        c.set_option(capi.OPT_SAMPLER, 1)
        c.reset()
        ctxs[mode] = c
    try:
        o.set_sampler_tables(t)
        oacc = np.zeros((h, w, 4), dtype="<f4")
        for sample in range(3):
            oacc, _, ost = o.render(cam, w, h, mb, sample_idx=sample, white_furnace=wf, radiance=oacc)
            for mode, c in ctxs.items():
                c.integrate_stepwise(mb) if mode == "stepwise" else c.integrate(mb)
                check_stats(c.frame_stats(), ost, mb)
                assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(oacc[..., :3])), (mode, sample)
        o.set_sampler_tables(None)
        plain, _, _ = o.render(cam, w, h, mb, sample_idx=0, white_furnace=wf)
        c = ctxs["fused"]
        c.set_option(capi.OPT_SAMPLER, 0); c.reset(); c.integrate(mb)      # switching back re-captures the frame graph
        assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(plain[..., :3]))
    finally:
        o.set_sampler_tables(None)
        for c in ctxs.values():
            c.destroy()


@pytest.mark.parametrize("n_tris", [1, 2])
def test_root_leaf_bvh_and_tiny_images(n_tris):
    """A BVH that is a single leaf, a 1x1 image, and a partition where one rank owns no row at all."""
    from tests.scenes_extra import single_leaf_scene
    sc = single_leaf_scene(n_tris)
    for (w, h) in [(1, 1), (33, 3)]:
        cam = default_camera(w, h)
        orad, _, ost = Oracle(sc).render(cam, w, h, 3)
        for traversal in (0, 1):
            c = capi.Context(w, h); c.upload_scene(sc); c.set_camera(cam); c.set_option(capi.OPT_TRAVERSAL, traversal)
            c.reset(); c.integrate(3)
            check_stats(c.frame_stats(), ost, 3)
            assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(orad[..., :3]))
            c.destroy()
    w, h = 33, 3
    out = np.zeros((h, w, 4), "<f4")
    for rank in range(4):                       # rank 3 owns zero rows
        c = capi.Context(w, h, rank=rank, world=4); c.upload_scene(sc); c.set_camera(default_camera(w, h))
        c.reset(); c.integrate(3); c.read_radiance(out); c.resolve(); c.destroy()
    assert np.array_equal(bits(out[..., :3]), bits(orad[..., :3]))


@pytest.mark.parametrize("name,w,h,mb", [("CornellBox", 320, 180, 8), ("ShaderBalls", 256, 144, 6)])
def test_shadow_pass_overlap_modes_are_equivalent(name, w, h, mb):
    """RT_OPT_OVERLAP 0 (in order), 1 (second stream) and 2 (shadow pass deferred into the next traversal kernel), with and
    without the frame graph / programmatic dependent launch, and with reads in the middle of a frame that force the
    deferred pass out early: same radiance, same counters."""
    sc = scene(name); cam = default_camera(w, h)
    o = Oracle(sc)
    want, _, ost = o.render(cam, w, h, mb)
    for overlap in (0, 1, 2):
        for graph, pdl in ((1, 1), (0, 1), (0, 0)):
            c = make_ctx(name, w, h)
            c.set_option(capi.OPT_FRAME_KERNEL, 0)           # the per-phase kernels (rt_integrate's default is the one-kernel frame)
            c.set_option(capi.OPT_OVERLAP, overlap); c.set_option(capi.OPT_GRAPH, graph); c.set_option(capi.OPT_PDL, pdl)
            c.reset(); c.integrate(mb)
            check_stats(c.frame_stats(), ost, mb)
            assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(want[..., :3])), (overlap, graph, pdl)
            c.destroy()
        # the per-virtual calls of the fused schedule, interrupted by taps
        c = make_ctx(name, w, h)
        c.set_option(capi.OPT_OVERLAP, overlap)
        c.reset(); c.generate_rays()
        partial, _, _ = o.render(cam, w, h, 2)
        for b in range(mb + 1):
            c.extend_shade(b)
            c.shadow_accumulate(b)
            if b == 2:                       # radiance after bounce 2 == a 2-bounce render
                assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(partial[..., :3])), overlap
            if b == 4:
                c.sync()
        c.advance_sample_count()
        check_stats(c.frame_stats(), ost, mb)
        assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(want[..., :3])), overlap
        c.destroy()


@pytest.mark.parametrize("name,w,h,mb", [("CornellBox", 300, 170, 6), ("ShaderBalls", 256, 144, 5)])
def test_point_lights_and_thin_lens_match_oracle(name, w, h, mb):
    """Five analytic lights (point + directional) and a thin-lens camera off the default pose: fused and stepwise vs the
    oracle (pinned on the same configuration in tests/test_oracle_vs_ref.py)."""
    from tests.scenes_extra import many_lights_scene
    sc = many_lights_scene(name)
    cam = default_camera(w, h, position=(0.15, -1.3, 0.9), aperture=0.04, focus_distance=1.7)
    o = Oracle(sc)
    oacc = np.zeros((h, w, 4), dtype="<f4")
    ctxs = []
    for stepwise in (False, True):
        c = capi.Context(w, h); c.upload_scene(sc); c.set_camera(cam); c.reset()
        ctxs.append((stepwise, c))
    for sample in range(2):
        oacc, ohits, ost = o.render(cam, w, h, mb, sample_idx=sample, radiance=oacc)
        for stepwise, c in ctxs:
            c.integrate_stepwise(mb) if stepwise else c.integrate(mb)
            check_stats(c.frame_stats(), ost, mb)
            assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(oacc[..., :3])), (stepwise, sample)
    for _, c in ctxs:
        c.destroy()


@pytest.mark.parametrize("case", ["zero_bounces", "all_miss", "inside_geometry"])
def test_degenerate_frames_match_oracle(case):
    """max_bounces = 0; a frame whose every primary ray misses (all later queues empty: persistent kernels with nothing to
    drain, merged traversal kernels with two empty queues); a camera inside closed geometry."""
    name, w, h, mb, kw = {"zero_bounces": ("CornellBox", 192, 128, 0, {}),
                          "all_miss": ("ShaderBalls", 160, 96, 4, {"position": (0.0, -30.0, 40.0), "pitch": 0.3}),
                          "inside_geometry": ("ShaderBalls", 160, 96, 4, {"position": (0.0, 0.0, 0.35), "pitch": 1.9})}[case]
    sc = scene(name); cam = default_camera(w, h, **kw)
    o = Oracle(sc)
    oacc = np.zeros((h, w, 4), dtype="<f4")
    ctxs = []
    for stepwise in (False, True):
        c = capi.Context(w, h); c.upload_scene(sc); c.set_camera(cam); c.reset()
        ctxs.append((stepwise, c))
    for sample in range(2):
        oacc, _, ost = o.render(cam, w, h, mb, sample_idx=sample, radiance=oacc)
        for stepwise, c in ctxs:
            c.integrate_stepwise(mb) if stepwise else c.integrate(mb)
            check_stats(c.frame_stats(), ost, mb)
            assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(oacc[..., :3])), (case, stepwise, sample)
    for _, c in ctxs:
        c.destroy()


def test_fuzzed_frames_match_oracle():
    """The seeded random configurations of tests/test_oracle_vs_ref.py (scenes, sizes, bounce counts, camera poses and lenses,
    axis-aligned views): fused schedule vs the oracle, two progressive samples each."""
    for name, w, h, mb, kw, wf in fuzz_configs():
        sc = scene(name); cam = default_camera(w, h, **kw)
        o = Oracle(sc)
        c = capi.Context(w, h); c.upload_scene(sc); c.set_camera(cam); c.set_option(capi.OPT_WHITE_FURNACE, int(wf)); c.reset()
        oacc = np.zeros((h, w, 4), dtype="<f4")
        for sample in range(2):
            oacc, _, ost = o.render(cam, w, h, mb, sample_idx=sample, white_furnace=wf, radiance=oacc)
            c.integrate(mb)
            check_stats(c.frame_stats(), ost, mb)
            assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(oacc[..., :3])), (name, w, h, mb, kw, wf, sample)
        c.destroy()


@pytest.mark.parametrize("name,w,h,mb", [("CornellBox", 333, 127, 8), ("ShaderBalls", 480, 270, 6), ("CornellBox_Dragon", 200, 112, 12), ("CornellBox", 37, 5, 3)])
def test_frame_kernel_matches_phase_kernels(name, w, h, mb):
    """RT_OPT_FRAME_KERNEL 1 (one persistent kernel per frame, CTA-private queues) vs 0 (one kernel per phase): radiance,
    counters and AOVs bit for bit, over three progressive samples, whole image and a 3-way scanline partition, with the BVH
    staged in shared memory and fetched through L1."""
    sc = scene(name); cam = default_camera(w, h)
    for world in (1, 3):
        for smem in (1, 0):
            imgs = {}
            for fk in (1, 0):
                rad = np.zeros((h, w, 4), "<f4"); stats = []; aovs = []
                for rank in range(world):
                    c = capi.Context(w, h, rank=rank, world=world)
                    c.set_option(capi.OPT_FRAME_KERNEL, fk); c.set_option(capi.OPT_SMEM_BVH, smem); c.set_option(capi.OPT_AOV_ALWAYS, 1)
                    c.upload_scene(sc); c.set_camera(cam); c.reset()
                    for _ in range(3):
                        c.integrate(mb)
                    c.read_radiance(rad)
                    stats.append(c.frame_stats()); aovs.append(c.read_aovs())
                    c.destroy()
                imgs[fk] = (rad, stats, aovs)
            assert np.array_equal(bits(imgs[1][0]), bits(imgs[0][0])), (world, smem)
            for a, b in zip(imgs[1][1], imgs[0][1]):
                for k in ("n_ext", "n_miss", "n_shadow", "n_cont", "n_unoccluded", "n_emissive_hits"):
                    assert np.array_equal(a[k][: mb + 1], b[k][: mb + 1]), (k, world, smem)
            for a, b in zip(imgs[1][2], imgs[0][2]):
                for x, y in zip(a, b):
                    assert np.array_equal(bits(np.asarray(x)), bits(np.asarray(y))), (world, smem)


@pytest.mark.parametrize("name,w,h,mb", [("ShaderBalls", 320, 180, 6), ("CornellBox_Dragon", 240, 135, 10)])
def test_top_of_tree_staging_is_bit_identical(name, w, h, mb):
    """RT_OPT_TOP_SMEM: scenes whose records do not fit shared memory stage the first k interior records (breadth-first top of the
    tree) with one TMA bulk copy per CTA; every k, in the per-phase kernels and in the one-kernel frame, gives the oracle's bits."""
    sc = scene(name); cam = default_camera(w, h)
    want, _, ost = Oracle(sc).render(cam, w, h, mb)
    for k in (8, 100, 640):
        for fk in (0, 1):
            c = make_ctx(name, w, h)
            c.set_option(capi.OPT_TOP_SMEM, k); c.set_option(capi.OPT_FRAME_KERNEL, fk)
            c.reset(); c.integrate(mb)
            check_stats(c.frame_stats(), ost, mb)
            assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(want[..., :3])), (k, fk)
            c.destroy()
    c = make_ctx(name, w, h)
    with pytest.raises(capi.RtError):
        c.set_option(capi.OPT_TOP_SMEM, 641)
    c.destroy()


@pytest.mark.parametrize("name,w,h,mb,fk", [("CornellBox", 203, 117, 6, 1), ("ShaderBalls", 320, 180, 5, 1), ("ShaderBalls", 257, 131, 7, 0)])
def test_fused_gather_delivers_the_frame(name, w, h, mb, fk):
    """rt_set_gather_target: the ranks' frame kernels push every pixel into rank 0's gather buffer the moment its path ends
    (misses in the shading phase, paths that end at a hit after their last shadow ray, survivors after the last round; the
    per-phase schedule copies its slab at the end).  Three ranks in one process share the buffer directly; after rt_gather_wait
    the buffer resolved through rt_resolve_gathered equals the single-context image, over three progressive samples."""
    sc = scene(name); cam = default_camera(w, h)
    world = 3
    one = capi.Context(w, h); one.upload_scene(sc); one.set_camera(cam); one.reset()
    parts = []
    for rank in range(world):
        c = capi.Context(w, h, rank=rank, world=world)
        c.set_option(capi.OPT_FRAME_KERNEL, fk)
        c.upload_scene(sc); c.set_camera(cam); c.reset()
        parts.append(c)
    buf, stride, total = parts[0].gather_buffer()
    assert total >= world * stride + 4 * world
    for c in parts:
        c.set_gather_target(buf, stride)
    for sample in range(3):
        one.integrate(mb)
        for c in reversed(parts):                # rank 0 last: its wait really waits for flags set on other streams
            c.integrate(mb)
        parts[0].gather_wait()
        got = parts[0].resolve_gathered(buf, stride)
        assert np.array_equal(bits(got), bits(one.resolve())), sample
    # turning it off again stops the pushes
    for c in parts:
        c.set_gather_target(None)
    with pytest.raises(capi.RtError):
        parts[0].gather_wait()
    for c in parts + [one]:
        c.destroy()


@pytest.mark.parametrize("name,w,h,mb", [("CornellBox", 203, 117, 6), ("ShaderBalls", 320, 180, 5)])
def test_multi_device_context_matches_single_device(name, w, h, mb):
    """rt_create_multi: ONE context over several devices (here the devices of the box, or device 0 listed three times when it has
    only one: three partitions time-share it), every call fanned out inside the library.  Radiance, counters, resolved image
    (parallel read-back and NVLink-gather presentation) and AOVs equal the single-device frame bit for bit."""
    sc = scene(name); cam = default_camera(w, h)
    n_dev = capi.device_count()
    devices = list(range(n_dev)) if n_dev >= 2 else [0, 0, 0]
    one = capi.Context(w, h); one.set_option(capi.OPT_AOV_ALWAYS, 1); one.upload_scene(sc); one.set_camera(cam); one.reset()
    many = capi.Context(w, h, devices=devices); many.set_option(capi.OPT_AOV_ALWAYS, 1); many.upload_scene(sc); many.set_camera(cam); many.reset()
    for sample in range(3):
        one.integrate(mb); many.integrate(mb)
    assert many.sample_count() == 3
    a, b = one.frame_stats(), many.frame_stats()
    for k in ("n_ext", "n_miss", "n_shadow", "n_cont", "n_unoccluded", "n_emissive_hits"):
        assert np.array_equal(a[k][: mb + 1], b[k][: mb + 1]), k
    assert np.array_equal(bits(one.read_radiance()), bits(many.read_radiance()))
    want = one.resolve()
    host = np.zeros((h, w, 4), "<f4"); capi.host_register(host)
    try:
        assert np.array_equal(bits(want), bits(many.resolve(host)))               # parallel read-back into a page-locked image
        many.set_option(capi.OPT_PRESENT, 1)
        host[:] = 0
        assert np.array_equal(bits(want), bits(many.resolve(host)))               # frames rendered before the option: peer copies to devices[0], resolve there
        one.integrate(mb); many.integrate(mb)                                      # a frame rendered WITH the option: pushed by the frame kernels (fused gather)
        want = one.resolve()
        host[:] = 0
        assert np.array_equal(bits(want), bits(many.resolve(host)))
        many.set_option(capi.OPT_PRESENT, 0)
        host[:] = 0
        many.resolve_async(host); many.resolve_wait()
        assert np.array_equal(bits(want), bits(host))
    finally:
        capi.host_unregister(host)
    for x, y in zip(one.read_aovs(), many.read_aovs()):
        assert np.array_equal(bits(x), bits(y))
    # the stepwise per-virtual calls fan out too
    one.reset(); many.reset()
    one.integrate_stepwise(mb); many.integrate_stepwise(mb)
    assert np.array_equal(bits(one.read_radiance()), bits(many.read_radiance()))
    with pytest.raises(capi.RtError):
        many.set_option(capi.OPT_DENOISER, 1)                # temporal reprojection needs the whole image on one device
    with pytest.raises(capi.RtError):
        many.stream_handle()                                 # single-device call
    one.destroy(); many.destroy()


def test_scene_reupload_and_camera_change_on_one_context():
    """UploadGPUData twice and SetCameraData between frames on the same context (the frame graph is re-captured when a
    launch argument changes, and only its per-frame constants are refreshed when the camera moves)."""
    w, h, mb = 200, 112, 5
    c = capi.Context(w, h)
    cams = [default_camera(w, h), default_camera(w, h, position=(0.3, -1.4, 1.2))]
    for name in ("CornellBox", "ShaderBalls", "CornellBox"):
        sc = scene(name); o = Oracle(sc)
        c.upload_scene(sc)
        for cam in cams:
            c.set_camera(cam); c.reset()
            acc = np.zeros((h, w, 4), dtype="<f4")
            for sample in range(2):
                c.integrate(mb)
                acc, _, ost = o.render(cam, w, h, mb, sample_idx=sample, radiance=acc)
                check_stats(c.frame_stats(), ost, mb)
                assert np.array_equal(bits(c.read_radiance()[..., :3]), bits(acc[..., :3])), (name, sample)
    c.destroy()


def test_error_behaviour():
    c = capi.Context(32, 32)
    with pytest.raises(capi.RtError):
        c.generate_rays()                     # no scene yet
    sc = dict(scene("CornellBox"))
    bad = dict(sc); bad["lights"] = sc["lights"][:0]
    with pytest.raises(capi.RtError):
        c.upload_scene(bad)                   # light.h:46 would divide by zero
    c.upload_scene(sc)
    with pytest.raises(capi.RtError):
        c.integrate(3)                        # no camera yet
    with pytest.raises(capi.RtError):
        c.set_option(capi.OPT_SAMPLER, 1)     # kBlueNoise without its tables: loud, not silent
    sob, scr, rank = synthetic_sampler_tables()
    bad_rank = rank.copy(); bad_rank[77] = 256
    with pytest.raises(capi.RtError):
        c.upload_sampler_tables(sob, scr, bad_rank)   # would index past the sobol table
    with pytest.raises(ValueError):
        c.upload_sampler_tables(sob[:100], scr, rank)
    c.upload_sampler_tables(sob, scr, rank)
    c.set_option(capi.OPT_SAMPLER, 1)
    with pytest.raises(capi.RtError):
        c.set_option(capi.OPT_SAMPLER, 2)
    c.destroy()
    c = capi.Context(32, 32, rank=1, world=2)
    with pytest.raises(capi.RtError):
        c.set_option(capi.OPT_DENOISER, 1)    # temporal reprojection needs the whole image on one GPU
    with pytest.raises(capi.RtError):
        capi.Context(70000, 16)               # pixel coordinates are packed in 16 + 16 bits
    c.destroy()
