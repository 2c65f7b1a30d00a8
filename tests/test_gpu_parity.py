"""GPU parity tests proper: the CUDA path, called through the C ABI (libcrtb200.so), against the CPU oracle on the same
inputs and against the committed reference fixtures.  Bar: bit-exact hit ids (mesh, triangle, t), bit-identical float RGB,
identical ray counts and identical traversal work; the north_star 8-bit tolerance (|d| <= 1 on >= 99.9 % of pixels, none
> 4) follows and is asserted too."""
import importlib
import os

import numpy as np
import pytest

import gi_oracle as gio
from conftest import PKG, ROOT, SMALL_SCENES, same_f32
from handoff_contexts import HandoffContexts

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(ROOT, "tests", "golden")
# hw14_small's 20 736 primary rays are more than the "capped" context's k_coop takes in one launch (4 736 walks on a B200:
# one per resident k_coop warp)
CAPPED_OVERFLOW = "hw14_small"


@pytest.fixture(scope="module")
def gpu(built):
    try:
        ctx = built.Context(0)
    except built.CrtError as e:  # fail loudly: the product has no CPU fallback
        pytest.fail(f"CUDA core unusable on a GPU box: {e}")
    yield ctx
    ctx.close()


def _covered(sf, rects, n):
    cov = np.zeros((sf.info.height, sf.info.width), bool)
    for i in range(n):
        r = rects[i]
        cov[r.row:r.row + r.height, r.col:r.col + r.width] = True
    return cov


def _assert_pixels(name, rgb, ref_rgb, q, ref_q):
    """Float RGB bit-identical (NaN == NaN) on every pixel -- refractive ones included, since the device evaluates the
    Fresnel powf exactly like glibc (csrc/crt_powf5.h) -- which implies the north_star 8-bit bar (|d| <= 1 on >= 99.9 %,
    none > 4), asserted separately so a float regression still reports how far the image moved."""
    d = np.abs(q.astype(np.int32) - ref_q.astype(np.int32)).max(axis=2)
    assert (d <= 1).mean() >= 0.999 and d.max() <= 4, f"{name}: 8-bit tolerance exceeded (max {d.max()})"
    same = same_f32(rgb, ref_rgb)
    assert same.all(), f"{name}: {(~same).sum()} float components differ (max |d| {np.nanmax(np.abs(rgb - ref_rgb))})"


@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_render_matches_oracle_and_golden(name, gpu, loaded, ob, crt):
    sf, flat, rects, n = loaded[name]
    gpu.upload(flat, keepalive=sf)
    opt = crt.make_options(rects=rects, n_rects=n, count_work=1)
    rgb, rgb8, hits, st = gpu.render(sf.camera(), opt, want_rgb8=True, want_hits=True)
    o_rgb, o_hits, o_st = ob.render(flat, sf.camera(), opt)
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    cov = _covered(sf, rects, n)
    # (i) hit ids: bit-exact, including t
    for ref_hits in (o_hits, g["hits"]):
        assert np.array_equal(hits["mesh"][cov], ref_hits["mesh"][cov])
        assert np.array_equal(hits["triangle"][cov], ref_hits["triangle"][cov])
        h = cov & (ref_hits["mesh"] >= 0)
        assert same_f32(hits["t"][h], ref_hits["t"][h]).all()
    # (ii) pixels
    _assert_pixels(name, rgb, o_rgb, rgb8, ob.quantize(o_rgb))
    _assert_pixels(name, rgb, g["rgb"], rgb8, g["ppm"])
    assert np.array_equal(rgb8, ob.quantize(rgb)), "device PPMColor quantiser differs from Color.cpp:12-16"
    # (iii) identical ray sets and, in visit-all counting mode, identical traversal work
    for k in ("rays_primary", "rays_shadow", "rays_reflection", "rays_refraction"):
        assert st[k] == o_st[k], (k, st[k], o_st[k])
    assert [st["rays_primary"], st["rays_shadow"], st["rays_reflection"], st["rays_refraction"]] == list(g["rays"])
    for k in ("node_tests_closest", "triangle_tests_closest", "node_tests_shadow", "triangle_tests_shadow"):
        assert st[k] == o_st[k], (k, st[k], o_st[k])


def test_uncovered_pixels_persist(gpu, loaded, crt):
    """colorBuffer persists across render() calls (RayTracer.h:69): uncovered pixels keep the previous frame."""
    sf, flat, rects, n = loaded["uncovered"]
    gpu.upload(flat, keepalive=sf)
    full, _, _, _ = gpu.render(sf.camera(), crt.make_options())
    part, _, _, _ = gpu.render(sf.camera(), crt.make_options(rects=rects, n_rects=n))
    assert same_f32(full, part).all()
    gpu.upload(flat, keepalive=sf)  # fresh buffer: uncovered pixels are (0,0,0), not background
    part2, _, _, _ = gpu.render(sf.camera(), crt.make_options(rects=rects, n_rects=n))
    cov = _covered(sf, rects, n)
    assert (~cov).any() and (part2[~cov] == 0).all()


def test_primary_rays_bit_exact(gpu, loaded, ob, crt, scenes_mod):
    sf, flat, _, _ = loaded["hw14_small"]
    gpu.upload(flat, keepalive=sf)
    for pos, rot in [((0.0, 0.3, 0.0), (1, 0, 0, 0, 1, 0, 0, 0, 1))] + scenes_mod.orbit_cameras(7)[1:4]:
        cam = crt.Camera.make(pos, rot)
        assert np.array_equal(gpu.generate_rays(cam).view(np.uint32), ob.generate_rays(flat, cam).view(np.uint32))


def test_trace_rays_random_and_nan(gpu, loaded, ob, crt):
    """RayTracer::trace / hasIntersection as plain queries, including NaN / axis-parallel / zero directions."""
    sf, flat, _, _ = loaded["hw11_room"]
    gpu.upload(flat, keepalive=sf)
    rng = np.random.default_rng(7)
    n = 20000
    rays = np.zeros((n, 6), np.float32)
    rays[:, 0:3] = rng.uniform(-1.9, 1.9, (n, 3)) + np.array([0, 0, -4.5])
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays[:, 3:6] = d
    rays[0:50, 3] = 0.0          # axis-parallel components (|d| < FLT_EPSILON branch of the slab test)
    rays[50:100, 4] = 0.0
    rays[100:110, 3:6] = np.nan  # NaN rays pass every test (SURVEY App. B-3)
    rays[110:120, 3:6] = 0.0
    for rt in (crt.RAY_PRIMARY, crt.RAY_REFLECTION):
        a, b = gpu.trace_rays(rays, rt), ob.trace_rays(flat, rays, rt)
        assert np.array_equal(a["mesh"], b["mesh"]) and np.array_equal(a["triangle"], b["triangle"])
        assert same_f32(a["t"], b["t"]).all()
    dist = rng.uniform(0.1, 6.0, n).astype(np.float32)
    assert np.array_equal(gpu.trace_rays(rays, crt.RAY_SHADOW, dist), ob.trace_rays(flat, rays, crt.RAY_SHADOW, dist))


def test_sharded_render_assembles_to_same_frame(gpu, loaded, crt):
    """Tile sharding (multi-GPU partition) emulated on one GPU: 3 shards rendered separately == full frame."""
    torch = pytest.importorskip("torch")
    sf, flat, _, _ = loaded["hw11_room"]
    gpu.upload(flat, keepalive=sf)
    full, _, _, _ = gpu.render(sf.camera(), crt.make_options())
    world = 3
    items = gpu.shard_items(world)
    slabs = torch.zeros((world, items, 3), dtype=torch.float32, device="cuda")
    for r in range(world):
        gpu.render_device(sf.camera(), crt.make_options(shard_index=r, shard_count=world), d_rgb=slabs[r].data_ptr(),
                          stream=torch.cuda.current_stream().cuda_stream)
    out = torch.zeros((sf.info.height, sf.info.width, 3), dtype=torch.float32, device="cuda")
    gpu.assemble_shards(slabs.data_ptr(), world, d_rgb=out.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().view(np.uint32), full.view(np.uint32))


def test_raytracer_mirror_and_ppm(gpu, loaded, ob, crt, tmp_path):
    """The C++ RayTracer mirror (render(path, options) + exportPPM) end to end: PPM byte-identical to the reference's."""
    sf, flat, rects, n = loaded["hw12_textures"]
    tracer = crt.RayTracer(sf)
    path = str(tmp_path / "out.ppm")
    rgb, st = tracer.render(path, mode=crt.MODE_B200_WAVEFRONT)
    g = np.load(os.path.join(GOLDEN, "hw12_textures.npz"))
    assert same_f32(rgb, g["rgb"]).all()
    assert np.array_equal(ob.read_ppm_p3(path), g["ppm"])
    tracer.close()


def test_chunked_frame_identical(gpu, loaded, crt):
    """A tiny queue budget forces the frame through several chunks; pixels and ray counts must not change."""
    sf, flat, _, _ = loaded["hw11_room"]
    gpu.upload(flat, keepalive=sf)
    a, _, _, sa = gpu.render(sf.camera(), crt.make_options())
    gpu.set_queue_budget(64 << 20)
    b, _, _, sb = gpu.render(sf.camera(), crt.make_options())
    gpu.set_queue_budget(16 << 30)
    assert same_f32(a, b).all()
    assert sa["rays_total"] == sb["rays_total"]


def test_small_chunks_with_moving_camera(gpu, loaded, crt, scenes_mod):
    """Chunks smaller than a row of tiles (tiny queue budget on a refractive scene, several chunk streams): band copies
    to the host would race between chunks sharing a 4-row band and leave stale rows of the PREVIOUS frame -- visible
    only when the camera moves between renders."""
    sf, flat, _, _ = loaded["hw11_room"]
    gpu.upload(flat, keepalive=sf)
    cams = [crt.Camera.make(p, r) for p, r in scenes_mod.orbit_cameras(12, radius=1.0, center_z=-2.0)[:4]]
    gpu.set_queue_budget(16 << 30)
    big = [gpu.render(cam, crt.make_options())[0].copy() for cam in cams]
    gpu.set_queue_budget(64 << 20)
    gpu.set_concurrency(6)
    small = [gpu.render(cam, crt.make_options())[0].copy() for cam in cams]
    gpu.set_queue_budget(16 << 30)
    for a, b in zip(big, small):
        assert same_f32(a, b).all()
    assert not same_f32(big[0], big[1]).all()  # the camera did move


@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_default_traversal_equals_literal_walk(name, gpu, loaded, crt):
    """traversal = 0 (default: conservative culling + tail hand-off, DESIGN.md 3.6 / 3.8) against traversal = 1 (the
    reference's literal visit-all itinerary): hit ids, t, float RGB and ray counts must be bit-identical on every scene,
    the NaN-triangle scene included (non-finite candidates only matter while no finite one exists, and nothing is
    culled until then).  The culled walk must also do less work than the literal one where there is anything to cull."""
    sf, flat, rects, n = loaded[name]
    gpu.upload(flat, keepalive=sf)
    a, _, ha, sa = gpu.render(sf.camera(), crt.make_options(rects=rects, n_rects=n, traversal=1, count_work=2), want_hits=True)
    b, _, hb, sb = gpu.render(sf.camera(), crt.make_options(rects=rects, n_rects=n, traversal=0, count_work=2), want_hits=True)
    assert same_f32(a, b).all()
    assert np.array_equal(ha["mesh"], hb["mesh"]) and np.array_equal(ha["triangle"], hb["triangle"])
    assert same_f32(ha["t"], hb["t"]).all()
    assert sa["rays_total"] == sb["rays_total"]
    assert sb["node_tests"] <= sa["node_tests"] and sb["triangle_tests"] <= sa["triangle_tests"]
    if name in ("hw14_small", "hw11_room", "hw07_scene0b"):
        assert sb["node_tests"] < sa["node_tests"]
        assert sa["shadow_rays_zero_term"] == 0
        if name != "hw11_room":  # (its diffuse surfaces are the room's walls: none is turned away from a light)
            assert sb["shadow_rays_zero_term"] > 0
    # count_work = 1 counts the reference's visit-all work whatever `traversal` says
    _, _, _, sc1 = gpu.render(sf.camera(), crt.make_options(rects=rects, n_rects=n, traversal=0, count_work=1))
    _, _, _, sc2 = gpu.render(sf.camera(), crt.make_options(rects=rects, n_rects=n, traversal=1, count_work=1))
    assert sc1["node_tests"] == sc2["node_tests"] and sc1["triangle_tests"] == sc2["triangle_tests"]


def test_dedup_does_less_work_than_visit_all_with_same_pixels(gpu, loaded, crt):
    """Production exact mode traverses a mesh once per ray even when several top-level leaves list it; count_work = 1
    reproduces the reference's repeated traversals (and its counters), count_work = 2 reports the real work."""
    sf, flat, rects, n = loaded["hw11_room"]
    gpu.upload(flat, keepalive=sf)
    a, _, _, visit_all = gpu.render(sf.camera(), crt.make_options(count_work=1))
    b, _, _, real = gpu.render(sf.camera(), crt.make_options(count_work=2))
    assert same_f32(a, b).all()
    assert real["node_tests"] < visit_all["node_tests"] and real["triangle_tests"] < visit_all["triangle_tests"]
    # more than 64 meshes: the visited-mesh set lives in shared memory instead of a 64-bit register, same effect
    sf, flat, rects, n = loaded["many_meshes"]
    assert flat.contents.n_meshes > 64
    gpu.upload(flat, keepalive=sf)
    a, _, _, visit_all = gpu.render(sf.camera(), crt.make_options(count_work=1))
    b, _, _, real = gpu.render(sf.camera(), crt.make_options(count_work=2, traversal=1))  # literal walk: only the de-duplication differs
    assert same_f32(a, b).all()
    assert real["node_tests"] < visit_all["node_tests"]


@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_production_path_matches_golden(name, gpu, loaded, crt):
    """count_work = 0 is what bench.py times: any-hit shadow rays, one walk per mesh, MODE 2 loops (thresholded node
    phase + warp-cooperative triangle phase).  Same bar as the counting mode: bit-identical to the reference fixtures."""
    sf, flat, rects, n = loaded[name]
    gpu.upload(flat, keepalive=sf)
    rgb, rgb8, hits, st = gpu.render(sf.camera(), crt.make_options(rects=rects, n_rects=n), want_rgb8=True, want_hits=True)
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    cov = _covered(sf, rects, n)
    assert np.array_equal(hits["mesh"][cov], g["hits"]["mesh"][cov]) and np.array_equal(hits["triangle"][cov], g["hits"]["triangle"][cov])
    h = cov & (g["hits"]["mesh"] >= 0)
    assert same_f32(hits["t"][h], g["hits"]["t"][h]).all()
    _assert_pixels(name, rgb, g["rgb"], rgb8, g["ppm"])
    assert [st["rays_primary"], st["rays_shadow"], st["rays_reflection"], st["rays_refraction"]] == list(g["rays"])


@pytest.fixture(scope="module")
def handoff(built):
    """Contexts with the tail hand-off forced or off (handoff_contexts.HANDOFF_ENV), created on first use."""
    hc = HandoffContexts(built)
    yield hc
    hc.close()


@pytest.mark.parametrize("which", ["all", "mid", "final_only", "off", "capped"])
@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_tail_handoff_matches_golden(name, which, handoff, loaded, crt):
    """k_coop explores a handed-off walk in a different order (a LIFO of subtrees, 32 boxes per iteration); by the nesting
    property the set of tested leaves is the same, and closest-hit candidates are put back into the reference's
    encounter order by their (leaf, reference) key -- so hit ids, t and every pixel stay bit-identical to the
    reference fixtures, with culling (traversal 0) and without (traversal 1 has no hand-off: literal walk).  "all" and "mid"
    run k_coop's early pass next to the traversal kernel plus the final pass behind it (small frames run on one stream),
    "final_only" the final pass alone.  "capped" asks to hand off every walk, but k_coop takes one walk per resident warp
    and launch: the lanes turned away keep walking in the traversal kernel."""
    ctx = handoff(which)
    sf, flat, rects, n = loaded[name]
    ctx.upload(flat, keepalive=sf)
    opt = crt.make_options(rects=rects, n_rects=n)
    rgb, rgb8, hits, st = ctx.render(sf.camera(), opt, want_rgb8=True, want_hits=True)
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    cov = _covered(sf, rects, n)
    assert np.array_equal(hits["mesh"][cov], g["hits"]["mesh"][cov]) and np.array_equal(hits["triangle"][cov], g["hits"]["triangle"][cov])
    h = cov & (g["hits"]["mesh"] >= 0)
    assert same_f32(hits["t"][h], g["hits"]["t"][h]).all()
    _assert_pixels(name, rgb, g["rgb"], rgb8, g["ppm"])
    assert [st["rays_primary"], st["rays_shadow"], st["rays_reflection"], st["rays_refraction"]] == list(g["rays"])
    if which in ("all", "final_only", "capped") and name not in ("empty_scene",):
        assert st["handoff_closest"] > 0  # (warps that fetched their rays before the queue ran dry poll it every 4th round)
    if which == "off":
        assert st["handoff_closest"] == 0 and st["handoff_shadow"] == 0
    if which == "capped" and name == CAPPED_OVERFLOW:
        # the capacity is reached: fewer walks are handed off than on the same frame with room for every walk
        handoff("all").upload(flat, keepalive=sf)
        _, _, _, st_all = handoff("all").render(sf.camera(), opt)
        assert st["handoff_closest"] < st_all["handoff_closest"], (st["handoff_closest"], st_all["handoff_closest"])


def test_tail_handoff_full_size_equals_literal_walk(gpu, handoff, built):
    """1920x1080 room with 196 608-triangle mirror and glass spheres, depth 5 (thousands of long walks on every level):
    default kernels, aggressive mid-flight hand-off and the literal walk must agree bit for bit."""
    import importlib
    bench_mod = importlib.import_module("bench")
    f, folder, kw, tex, depth = bench_mod.ensure_scene("hw11_room_128", {})
    sf = built.SceneFile(f, folder)
    flat = sf.flatten()
    outs = []
    for ctx, trav in ((gpu, 1), (gpu, 0), (handoff("mid"), 0)):
        ctx.upload(flat, keepalive=sf)
        rgb, _, hits, st = ctx.render(sf.camera(), built.make_options(max_depth=depth, traversal=trav), want_hits=True)
        outs.append((rgb, hits, st))
    for k in (1, 2):
        assert np.array_equal(outs[0][1]["triangle"], outs[k][1]["triangle"]) and np.array_equal(outs[0][1]["mesh"], outs[k][1]["mesh"])
        assert same_f32(outs[0][1]["t"], outs[k][1]["t"]).all()
        assert same_f32(outs[0][0], outs[k][0]).all()
        assert outs[0][2]["rays_total"] == outs[k][2]["rays_total"]


def test_trees_that_do_not_nest_take_the_literal_walk(gpu, handoff, built, scene_dir, ob, crt):
    """Culling and the order-free walk of k_coop are only equivalent to the reference's walk when every child box lies
    inside its parent's.  A caller may upload any tree through the C ABI: shrink one inner box so its children stick out
    -> the library must fall back to the literal walk, i.e. still agree with the oracle run on the very same (odd) tree.
    GI frames too, even in a context that would hand off every walk."""
    sf = built.SceneFile("hw14_small.crtscene", scene_dir)
    flat = sf.flatten()
    s = flat.contents
    big = max(range(s.n_meshes), key=lambda m: s.meshes[m].n_nodes)
    root = s.mesh_nodes[s.meshes[big].first_node]
    assert root.leaf_count == 0
    root.box_min[0] += 0.25 * (root.box_max[0] - root.box_min[0])  # children keep the old min.x: no longer nested
    gpu.upload(flat, keepalive=sf)
    rgb, _, hits, st = gpu.render(sf.camera(), crt.make_options(), want_hits=True)
    o_rgb, o_hits, o_st = ob.render(flat, sf.camera(), crt.make_options())
    assert np.array_equal(hits["mesh"], o_hits["mesh"]) and np.array_equal(hits["triangle"], o_hits["triangle"])
    assert same_f32(rgb, o_rgb).all()
    assert st["rays_total"] == o_st["rays_total"]
    _, _, _, a = gpu.render(sf.camera(), crt.make_options(count_work=2, traversal=0))
    _, _, _, b = gpu.render(sf.camera(), crt.make_options(count_work=2, traversal=1))
    # nothing was culled: the closest-hit walks execute the literal walk's box tests one for one; the shadow kernel
    # differs only by the rays whose light term is exactly zero (answered without a walk whatever the tree looks like)
    assert a["node_tests_closest"] == b["node_tests_closest"]
    assert a["triangle_tests_closest"] == b["triangle_tests_closest"]
    assert a["handoff_closest"] == a["handoff_shadow"] == 0
    assert a["shadow_rays_zero_term"] > 0 and b["shadow_rays_zero_term"] == 0
    assert a["node_tests_shadow"] < b["node_tests_shadow"]
    ctx = handoff("all")
    ctx.upload(flat, keepalive=sf)
    smp = crt.Sampling.make(gi_samples=1, rays_per_pixel=2, seed=11)
    opt = crt.make_options(max_depth=5)
    ctx.set_sampling(smp)
    g_rgb, _, g_hits, g = ctx.render(sf.camera(), opt, want_hits=True)
    ctx.set_sampling(None)
    o_rgb, o_hits, o_st = gio.render_sampled(flat, sf.camera(), opt, smp)
    assert same_f32(g_rgb, o_rgb).all(), f"{(~same_f32(g_rgb, o_rgb)).sum()} components differ"
    assert np.array_equal(g_hits["mesh"], o_hits["mesh"]) and np.array_equal(g_hits["triangle"], o_hits["triangle"])
    assert [g[k] for k in ("rays_primary", "rays_shadow", "rays_reflection", "rays_refraction")] == \
        [o_st[k] for k in ("rays_primary", "rays_shadow", "rays_reflection", "rays_refraction")]
    assert g["handoff_closest"] == g["handoff_shadow"] == 0


def test_multi_gpu_context_matches_single(gpu, built, loaded, crt):
    """crtb200_create_multi: the frame's tiles are dealt over the GPUs of the context, every GPU stores straight into the
    primary's frame (peer-mapped memory).  Same calls, same results as one GPU: float RGB, PPMColor bytes, hits, ray
    counts -- with every visible GPU, and with one GPU listed three times (three tile shards on one device)."""
    n = core_device_count(crt)
    lists = [[0, 0, 0]] + ([list(range(n))] if n > 1 else [])
    for ids in lists:
        multi = crt.Context(ids)
        assert multi.devices() == ids
        for name in ("hw11_room", "uncovered", "hw14_small", "one_pixel"):
            sf, flat, rects, nr = loaded[name]
            gpu.upload(flat, keepalive=sf)
            multi.upload(flat, keepalive=sf)
            opt = crt.make_options(rects=rects, n_rects=nr)
            a, a8, ha, sa = gpu.render(sf.camera(), opt, want_rgb8=True, want_hits=True)
            b, b8, hb, sb = multi.render(sf.camera(), opt, want_rgb8=True, want_hits=True)
            assert same_f32(a, b).all(), (ids, name)
            assert np.array_equal(a8, b8)
            cov = _covered(sf, rects, nr)
            assert np.array_equal(ha["mesh"][cov], hb["mesh"][cov]) and np.array_equal(ha["triangle"][cov], hb["triangle"][cov])
            for k in ("rays_primary", "rays_shadow", "rays_reflection", "rays_refraction"):
                assert sa[k] == sb[k], (ids, name, k)
        # batched animation through the multi-GPU context == per-camera renders on one GPU
        sf, flat, _, _ = loaded["hw14_small"]
        gpu.upload(flat, keepalive=sf)
        multi.upload(flat, keepalive=sf)
        cams = [crt.Camera.make(p, r) for p, r in importlib.import_module(PKG + ".scenes").orbit_cameras(5, radius=5.12, center_z=-4.0)]
        frames, _, _ = multi.render_frames(cams, crt.make_options())
        for k, cam in enumerate(cams):
            one, _, _, _ = gpu.render(cam, crt.make_options())
            assert same_f32(frames[k], one).all()
        multi.close()


def core_device_count(crt):
    import ctypes as C
    n = C.c_int(0)
    assert crt.core().crtb200_device_count(C.byref(n)) == 0
    return n.value


def test_context_error_is_per_context(gpu, built, crt):
    other = crt.Context(0)
    with pytest.raises(crt.CrtError):
        other.render(crt.Camera.make(), crt.make_options())  # no scene uploaded
    assert "no scene" in other.last_error()
    assert "no scene" not in gpu.last_error()
    other.close()


def test_raytracer_refuses_linear_scan_modes(loaded, crt):
    """NoOptimization / Regions / Buckets* / AABB* use RayTracer::trace's linear scan in the reference (RayTracer.cpp:
    459-505): other tie and NaN rules than the tree path.  The mirror renders the tree modes only and says so."""
    sf, flat, rects, n = loaded["hw07_scene0"]
    tracer = crt.RayTracer(sf)
    for mode in (0, 1, 2, 3, 4, 5, 6):
        with pytest.raises(crt.CrtError, match="tree modes"):
            tracer.render("", mode=mode)
    a, _ = tracer.render("", mode=crt.MODE_BVH_BUCKETS_THREADPOOL)
    b, _ = tracer.render("", mode=crt.MODE_B200_WAVEFRONT)
    c, _ = tracer.render("", mode=crt.MODE_B200_WAVEFRONT, literal=True)
    assert same_f32(a, b).all() and same_f32(a, c).all()
    tracer.close()


def test_assemble_keeps_uncovered_pixels(gpu, loaded, crt):
    """Sharded render of a rectangle list that leaves pixels uncovered: crtb200_assemble_shards must not overwrite them."""
    torch = pytest.importorskip("torch")
    sf, flat, rects, n = loaded["uncovered"]
    gpu.upload(flat, keepalive=sf)
    full, _, _, _ = gpu.render(sf.camera(), crt.make_options(rects=rects, n_rects=n))
    world = 2
    items = gpu.shard_items(world)
    slabs = torch.zeros((world, items, 3), dtype=torch.float32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for r in range(world):
        gpu.render_device(sf.camera(), crt.make_options(rects=rects, n_rects=n, shard_index=r, shard_count=world), d_rgb=slabs[r].data_ptr(), stream=st)
    out = torch.full((sf.info.height, sf.info.width, 3), 7.0, dtype=torch.float32, device="cuda")
    gpu.assemble_shards(slabs.data_ptr(), world, d_rgb=out.data_ptr(), stream=st)
    torch.cuda.synchronize()
    out = out.cpu().numpy()
    cov = _covered(sf, rects, n)
    assert same_f32(out[cov], full[cov]).all() and (out[~cov] == 7.0).all()


@pytest.mark.parametrize("name", ["hw11_room", "hw14_small", "uncovered", "many_meshes"])
def test_reference_binary_with_b200_binding_writes_the_same_ppm(name, built, ob, scene_dir, tmp_path):
    """INTEGRATION.md section B compiled for real: oracle/_ref/crt_ref_b200 = the UNMODIFIED reference's SceneParser,
    RayTracer constructor (AABB + KDTree::build) and exportPPM around crtb200_render (oracle/ref_b200_binding.cpp flattens
    the reference's own Scene / KDTree objects into the C ABI).  Its PPM must equal, byte for byte, the one the reference
    writes when it renders on the CPU (crt_ref), for one GPU and for three tile shards."""
    import subprocess
    exe = os.path.join(ROOT, "oracle", "_ref", "crt_ref_b200")
    if not (os.path.exists(exe) and ob.have_reference(False)):
        pytest.skip("needs oracle/_ref, compiled from the original program's C++ sources (oracle/build_ref.sh), "
                    "which are not part of this repository")
    ref = ob.run_reference(name + ".crtscene", scene_dir, str(tmp_path / "cpu"), hits=False)
    want = open(ref["ppm_path"], "rb").read()
    for devices in (1, 3):  # 3 > visible GPUs on a one-GPU box is refused by crtb200_create_multi ...
        out = str(tmp_path / f"gpu{devices}.ppm")
        r = subprocess.run([exe, name + ".crtscene", scene_dir, out, "--devices", str(devices)], capture_output=True, text=True, timeout=600)
        if devices > 1 and r.returncode != 0 and "no such CUDA device" in r.stderr:
            continue  # ... which is the right answer there
        assert r.returncode == 0, r.stderr[-2000:]
        assert open(out, "rb").read() == want, f"{name}: PPM of the reference + B200 binding differs from the reference's own"


def test_shards_written_in_place_make_the_same_frame(gpu, loaded, crt):
    """options.shard_full_frame: each tile shard is stored at its place in ONE full frame (what the ranks of a multi-
    process run do into rank 0's IPC-mapped frame); three shards == the unsharded frame, f32 and PPMColor bytes."""
    torch = pytest.importorskip("torch")
    sf, flat, _, _ = loaded["hw11_room"]
    gpu.upload(flat, keepalive=sf)
    full, full8, _, _ = gpu.render(sf.camera(), crt.make_options(), want_rgb8=True)
    H, W = sf.info.height, sf.info.width
    out = torch.zeros((H, W, 3), dtype=torch.float32, device="cuda")
    out8 = torch.zeros((H, W, 3), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for r in range(3):
        gpu.render_device(sf.camera(), crt.make_options(shard_index=r, shard_count=3, shard_full_frame=True),
                          d_rgb=out.data_ptr(), d_rgb8=out8.data_ptr(), stream=st)
    torch.cuda.synchronize()
    assert same_f32(out.cpu().numpy(), full).all()
    assert np.array_equal(out8.cpu().numpy(), full8)


def test_shards_stored_into_pinned_host_memory_make_the_same_frame(gpu, loaded, crt):
    """The e2e leg of an N-GPU frame: every rank's store kernel writes its tiles straight into ONE pinned host frame
    (multigpu.SharedHostFrame: mapped host memory, zero-copy over PCIe).  Here: three shards of one GPU into a pinned
    host tensor == the unsharded frame."""
    torch = pytest.importorskip("torch")
    sf, flat, _, _ = loaded["hw14_small"]
    gpu.upload(flat, keepalive=sf)
    full, _, _, _ = gpu.render(sf.camera(), crt.make_options())
    H, W = sf.info.height, sf.info.width
    host = torch.zeros((H, W, 3), dtype=torch.float32).pin_memory()
    st = torch.cuda.current_stream().cuda_stream
    for r in range(3):
        # (pinned memory allocated by the CUDA runtime is mapped; under unified addressing its device address is its host address)
        gpu.render_device(sf.camera(), crt.make_options(shard_index=r, shard_count=3, shard_full_frame=True),
                          d_rgb=host.data_ptr(), stream=st)
    torch.cuda.synchronize()
    assert same_f32(host.numpy(), full).all()


def test_shared_host_frame_single_rank(gpu, built, loaded, crt):
    """multigpu.SharedHostFrame + PeerStoreRenderer.render_to_host with a one-rank process group (the collective plumbing,
    the shared-memory segment, cudaHostRegister): the host frame equals the frame of a plain render."""
    torch = pytest.importorskip("torch")
    import socket
    import torch.distributed as dist
    mg = importlib.import_module(PKG + ".multigpu")
    if dist.is_initialized():
        pytest.skip("a process group already exists in this process")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1)
    try:
        sf, flat, _, _ = loaded["hw11_room"]
        gpu.upload(flat, keepalive=sf)
        full, _, _, _ = gpu.render(sf.camera(), crt.make_options())
        H, W = sf.info.height, sf.info.width
        dev = torch.device("cuda", 0)
        peer = mg.PeerStoreRenderer(crt, gpu, torch, dist, dev, W, H)
        shared = mg.SharedHostFrame(torch, dist, W, H)
        assert shared.usable
        shared.array[:] = 0
        peer.render_to_host(sf.camera(), shared)
        torch.cuda.synchronize()
        assert same_f32(np.array(shared.array), full).all()
        shared.close()
        peer.close()
    finally:
        dist.destroy_process_group()
