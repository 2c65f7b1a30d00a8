"""GPU: crtb200_upload_geometry, the device KD build (csrc/crt_build.cuh, DESIGN.md 3.11).  The trees it builds must be
the host builder's node for node, and it must leave the context exactly as crtb200_upload_scene of those trees does:
the device scene state bit for bit (nodes, references, node ranges, culling margins, the nesting flag) and therefore
every frame."""
import ctypes as C
import importlib
import os

import numpy as np
import pytest

import kd_build_oracle as kb
from conftest import ROOT, SMALL_SCENES, same_f32
from test_gpu_fullsize import _assert_frame_is_reference, _load, _reference_frame

pytestmark = pytest.mark.gpu
ERR_ARG, ERR_STATE, ERR_SCENE = -1, -3, -5
# timings, and the hand-off counts, which depend on when a queue runs dry (DESIGN.md 3.8)
TIMING = ("device_ms", "closest_ms", "shadow_ms", "total_ms", "coop_closest_ms", "coop_shadow_ms", "handoff_closest", "handoff_shadow")


@pytest.fixture(scope="module")
def gpu(built):
    ctx = built.Context(0)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def bench_mod():
    return importlib.import_module("bench")


def assert_layout_equal(a, b):
    for k in ("nodes", "leaf_refs", "top_refs", "meshes"):
        assert a[k].shape == b[k].shape and np.array_equal(a[k], b[k]), k
    assert (a["top_begin"], a["top_end"], a["nested_ok"]) == (b["top_begin"], b["top_end"], b["nested_ok"])


def _counts(st):
    return {k: v for k, v in st.items() if k not in TIMING}


def _frames(ctx, crt, sf, rects, n):
    """Unsampled frames in the default traversal, traversal 1, count_work 1 and 2; GI frames in two sampling
    configurations: (rgb, hits, counts) each."""
    out = []
    for kw in (dict(), dict(traversal=1), dict(count_work=1), dict(count_work=2)):
        rgb, _, hits, st = ctx.render(sf.camera(), crt.make_options(rects=rects, n_rects=n, **kw), want_hits=True)
        out.append((rgb, hits, _counts(st)))
    for smp in (crt.Sampling.make(gi_samples=2, rays_per_pixel=2, seed=11), crt.Sampling.make(gi_samples=1, rays_per_pixel=3, seed=5)):
        ctx.set_sampling(smp)
        rgb, _, hits, st = ctx.render(sf.camera(), crt.make_options(rects=rects, n_rects=n), want_hits=True)
        out.append((rgb, hits, dict(_counts(st), **ctx.sampling_stats())))
    ctx.set_sampling(None)
    return out


def _assert_frames_equal(a, b, ignore=()):
    for (ra, ha, sa), (rb, hb, sb) in zip(a, b):
        assert same_f32(ra, rb).all()
        assert np.array_equal(ha["mesh"], hb["mesh"]) and np.array_equal(ha["triangle"], hb["triangle"])
        assert same_f32(ha["t"], hb["t"]).all()
        assert {k: v for k, v in sa.items() if k not in ignore} == {k: v for k, v in sb.items() if k not in ignore}


@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_small_scene_trees_state_and_frames(name, gpu, loaded, built):
    """1-3: trees equal the host builder's, device state equals upload_scene's, frames and statistics equal, and the
    unsampled frame equals the golden fixture."""
    sf, flat, rects, n = loaded[name]
    gpu.upload(flat, keepalive=sf)
    host_layout = gpu.debug_scene_layout()
    host_frames = _frames(gpu, built, sf, rects, n)
    gpu.upload_geometry(sf.flatten(trees=False), keepalive=sf)
    t = gpu.scene_trees()
    kb.assert_trees_equal(kb.device_trees(t), kb.host_trees(flat))
    host_meshes = kb.scene_arrays(flat)["meshes"]
    for f in ("material", "first_triangle", "n_triangles", "first_vertex", "n_vertices"):
        assert np.array_equal(t["meshes"][f], host_meshes[f]), f
    assert t["peak_scratch_bytes"] > 0 and t["build_ms"] > 0
    assert_layout_equal(gpu.debug_scene_layout(), host_layout)
    dev_frames = _frames(gpu, built, sf, rects, n)
    _assert_frames_equal(dev_frames, host_frames)
    g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    assert same_f32(dev_frames[0][0], g["rgb"]).all()
    assert [dev_frames[0][2][k] for k in ("rays_primary", "rays_shadow", "rays_reflection", "rays_refraction")] == list(g["rays"])


def _small_triangles(rng, n, lo, hi, size):
    """n triangles of extent <= size around uniform centres in [lo, hi]^3: small against the scene, so that the trees
    stay small (triangles that overlap every split plane make the reference's tree grow as 2^depth)."""
    c = rng.uniform(lo, hi, (n, 1, 3))
    return (c + rng.uniform(0, size, (n, 3, 3))).astype(np.float32).reshape(-1, 3)


def _edge_scenes():
    """(name, vertex positions, triangles, mesh ranges) of scenes that cannot be written as .crtscene files."""
    rng = np.random.default_rng(5)
    out = []
    # -0.0 and +0.0, in both orders, on box extremes: two one-triangle meshes, then 40 triangles on the grid {0, 0.5, 1}^3
    # whose zero coordinates carry random signs, and the same triangles in reverse order
    head = np.array([[-0.0, 0.0, -0.0], [1, 1, 1], [0.5, -0.0, 0.0], [0.0, -0.0, 0.0], [1, 1, 1], [-0.0, 0.5, -0.0]], np.float32)
    g = rng.integers(0, 3, (40, 1, 3)) * 0.5 + rng.integers(0, 2, (40, 3, 3)) * 0.125
    g = np.where(g == 0, np.where(rng.integers(0, 2, g.shape) == 1, -0.0, 0.0), g).astype(np.float32).reshape(-1, 3)
    vp = np.concatenate([head, g])
    tv = np.concatenate([np.arange(6).reshape(2, 3), 6 + np.arange(120).reshape(40, 3), 6 + np.arange(120).reshape(40, 3)[::-1]])
    out.append(("signed_zeros", vp, tv, [(0, 1), (1, 1), (2, 40), (42, 40)]))
    p = _small_triangles(rng, 30, -2, 2, 0.3)
    p[4, 1] = np.nan
    p[9:12] = np.nan
    out.append(("nan", p, np.arange(90).reshape(30, 3), [(0, 30)]))
    out.append(("empty_mesh", _small_triangles(rng, 20, -2, 2, 0.3), np.arange(60).reshape(20, 3), [(0, 10), (10, 0), (10, 10)]))
    vp, tv = kb.coincident_triangles(12)
    out.append(("coincident", vp, tv, [(0, 13)]))
    p = np.concatenate([_small_triangles(rng, 3, c - 0.2, c + 0.2, 0.1) for c in rng.uniform(-3, 3, 70)])
    out.append(("many_meshes", p, np.arange(70 * 9).reshape(-1, 3), [(3 * i, 3) for i in range(70)]))
    out.append(("zero_meshes", np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32), []))
    p = _small_triangles(rng, 40, -2, 2, 0.3)
    p[:, 1] = 0.25
    out.append(("planar", p, np.arange(120).reshape(40, 3), [(0, 40)]))
    p = np.clip(_small_triangles(rng, 20, -3.3e38, 3.3e38, 1e37), -3.4e38, 3.4e38).astype(np.float32)
    p[0] = [3.4028235e38, -3.4028235e38, 3.4028235e38]
    out.append(("near_flt_max", p, np.arange(60).reshape(20, 3), [(0, 12), (12, 8)]))
    return out


EDGE = _edge_scenes()


@pytest.mark.parametrize("case", EDGE, ids=[e[0] for e in EDGE])
def test_edge_scene_built_from_arrays(case, gpu, built):
    """4: trees equal the restatement's; device state equals upload_scene of the restatement's trees."""
    name, vp, tv, ranges = case
    exp = kb.build_scene_trees(vp, tv, ranges)
    geo = kb.ArrayScene(built, vp, tv, ranges)
    gpu.upload_geometry(geo.ptr, keepalive=geo)
    kb.assert_trees_equal(kb.device_trees(gpu.scene_trees()), exp)
    dev = gpu.debug_scene_layout()
    cam = built.Camera.make((0.0, 0.0, 5.0))
    rgb_dev, _, hits_dev, _ = gpu.render(cam, built.make_options(), want_hits=True)
    host = kb.ArrayScene(built, vp, tv, ranges, trees=exp)
    gpu.upload(host.ptr, keepalive=host)
    assert_layout_equal(dev, gpu.debug_scene_layout())
    rgb_host, _, hits_host, _ = gpu.render(cam, built.make_options(), want_hits=True)
    assert same_f32(rgb_dev, rgb_host).all() and np.array_equal(hits_dev["triangle"], hits_host["triangle"])
    if name == "empty_mesh":
        assert not dev["nested_ok"]
    if name == "coincident":
        assert np.sort(exp["mesh_nodes"]["leaf_count"])[-1] == 13


def test_determinism_and_multi_gpu_replicas(gpu, loaded, built):
    """5: two uploads give identical state; every replica of Context([0, 0, 0]) equals the single-GPU context's, and
    so do its frames."""
    sf, flat, rects, n = loaded["hw14_small"]
    geo = sf.flatten(trees=False)
    gpu.upload_geometry(geo, keepalive=sf)
    a = gpu.debug_scene_layout()
    gpu.upload_geometry(geo, keepalive=sf)
    assert_layout_equal(a, gpu.debug_scene_layout())
    one = _frames(gpu, built, sf, rects, n)
    multi = built.Context([0, 0, 0])
    try:
        multi.upload_geometry(geo, keepalive=sf)
        for d in range(3):
            assert_layout_equal(multi.debug_scene_layout(d), a)
        kb.assert_trees_equal(kb.device_trees(multi.scene_trees()), kb.host_trees(flat))
        # every GPU of the context launches its own kernels for its tile shard: the launch count is per context
        _assert_frames_equal(_frames(multi, built, sf, rects, n), one, ignore=("kernel_launches",))
    finally:
        multi.close()


def test_errors(built, loaded):
    """6: tree arrays given, a vertex index out of range, read-back without a device-built scene, and the end of a
    progressive session."""
    core = built.core()
    ctx = built.Context(0)
    try:
        t = built.Trees()
        assert core.crtb200_scene_trees(ctx._h, C.byref(t)) == ERR_STATE  # before any upload
        sf, flat, rects, n = loaded["hw11_room"]
        assert core.crtb200_upload_geometry(ctx._h, flat) == ERR_ARG  # the host-built trees are attached
        ctx.upload(flat, keepalive=sf)
        assert core.crtb200_scene_trees(ctx._h, C.byref(t)) == ERR_STATE  # after upload_scene
        vp, tv = kb.coincident_triangles(2)
        bad = tv.copy()
        bad[1, 2] = 99
        fn = np.zeros((3, 3), np.float32)  # the helper cannot compute normals of a triangle whose vertex does not exist
        s = kb.ArrayScene(built, vp, bad, [(0, 3)], face_normals=fn)
        assert core.crtb200_upload_geometry(ctx._h, s.ptr) == ERR_SCENE
        s = kb.ArrayScene(built, vp, bad, [(0, 3)], trees=kb.build_scene_trees(vp, tv, [(0, 3)]), face_normals=fn)
        assert core.crtb200_upload_scene(ctx._h, s.ptr) == ERR_SCENE
        ctx.upload_geometry(sf.flatten(trees=False), keepalive=sf)
        p = ctx.progressive(sf.camera(), built.make_options(rects=rects, n_rects=n), built.Sampling.make())
        p.step(1)
        ctx.upload_geometry(sf.flatten(trees=False), keepalive=sf)
        assert core.crtb200_accum_step(ctx._h, 1, None) == ERR_STATE
        ctx.upload(flat, keepalive=sf)
        assert core.crtb200_scene_trees(ctx._h, C.byref(t)) == ERR_STATE
    finally:
        ctx.close()


@pytest.mark.parametrize("name", ["hw14_dragon_class", "synthetic_10M"])
def test_full_size(name, gpu, built, bench_mod, scenes_mod):
    """7: at BASELINE.json's sizes the trees equal the host builder's, the device state equals upload_scene's, and the
    frame is the stored one (sampled pixels, whole-frame digests, ray counts)."""
    sf, f, folder, tex, depth = _load(bench_mod, built, name)
    cam = sf.camera()
    if name == "synthetic_10M":
        pos, rot = scenes_mod.orbit_cameras(60, radius=5.12, center_z=-3.0)[7]
        cam = built.Camera.make(pos, rot)
    ref = _reference_frame(name, sf, f, folder, cam)
    flat = sf.flatten()
    gpu.upload(flat, keepalive=sf)
    host_layout = gpu.debug_scene_layout()
    gpu.upload_geometry(sf.flatten(trees=False), keepalive=sf)
    kb.assert_trees_equal(kb.device_trees(gpu.scene_trees()), kb.host_trees(flat))
    assert_layout_equal(gpu.debug_scene_layout(), host_layout)
    del host_layout
    rects, n = sf.rects(mode=built.MODE_BVH_BUCKETS_THREADPOOL)
    rgb, rgb8, hits, st = gpu.render(cam, built.make_options(max_depth=depth, rects=rects, n_rects=n), want_rgb8=True, want_hits=True)
    _assert_frame_is_reference(ref, rgb, rgb8, hits, st)
    sf.close()
