"""Caller-supplied ray batches on the GPU (crtb200_trace_rays_device, Context.trace; DESIGN.md 3.12): the production walk
(culling, tail hand-off to k_coop) answers caller rays held in CUDA tensors bit for bit as the CPU oracle's
crt_oracle_trace_rays does -- closest hits as RayTracer::trace, shadow queries as the non-GI RayTracer::hasIntersection --
for any direction length, under every hand-off setting, on several GPUs and on non-default streams, without touching the
context's frame state.  The last tests need no GPU: the C ABI surface of the feature."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, SMALL_SCENES, same_f32
from handoff_contexts import HANDOFF, HandoffContexts

ERR_ARG, ERR_STATE = -1, -3
CLOSEST_TYPES = ("RAY_PRIMARY", "RAY_REFLECTION", "RAY_REFRACTION")


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def gpu(built):
    ctx = built.Context(0)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def handoff(built):
    hc = HandoffContexts(built)
    yield hc
    hc.close()


def _box(flat):
    s = flat.contents
    if s.n_vertices == 0:
        return np.array([-1.0, -1.0, -1.0]), np.array([1.0, 1.0, 1.0]), np.zeros((1, 3))
    v = np.ctypeslib.as_array(s.vertex_position, shape=(3 * s.n_vertices,)).reshape(-1, 3).astype(np.float64)
    return v.min(axis=0), v.max(axis=0), v


def caller_rays(flat, n, seed):
    """Origins in and around the scene box; half the directions aimed at vertices (hits), half random; axis-parallel
    components, zero / NaN / inf directions and non-unit directions (x1e-3, x0.5, x3) in fixed slices."""
    rng = np.random.default_rng(seed)
    lo, hi, v = _box(flat)
    ext = np.maximum(hi - lo, 1e-3)
    o = rng.uniform(lo - 0.2 * ext, hi + 0.2 * ext, (n, 3))
    d = rng.normal(size=(n, 3))
    aim = rng.random(n) < 0.5
    d[aim] = v[rng.integers(0, len(v), aim.sum())] - o[aim]
    d /= np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-30)
    rays = np.concatenate([o, d], axis=1).astype(np.float32)
    k = n // 16
    rays[0:k, 3] = 0.0                       # axis-parallel components (|d| < FLT_EPSILON branch of the slab test)
    rays[k:2 * k, 4] = 0.0
    rays[2 * k:2 * k + 8, 3:5] = 0.0         # parallel to two axes
    rays[2 * k + 8:2 * k + 16, 3:6] = 0.0    # zero direction
    rays[2 * k + 16:2 * k + 24, 3:6] = np.nan
    rays[2 * k + 24:2 * k + 28, 3] = np.inf
    rays[3 * k:4 * k, 3:6] *= np.float32(1e-3)  # non-unit directions
    rays[4 * k:5 * k, 3:6] *= np.float32(0.5)
    rays[5 * k:6 * k, 3:6] *= np.float32(3.0)
    diag = float(np.linalg.norm(ext))
    dist = rng.uniform(0.05, 1.5 * diag, n).astype(np.float32)
    dist[0:16] = 0.0
    dist[16:32] = -1.0
    dist[32:40] = np.nan
    dist[40:48] = np.inf
    return rays, dist


def _same_hits(h, ref, what=""):
    m, tri, t = (x.cpu().numpy() for x in (h.mesh, h.triangle, h.t))
    assert np.array_equal(m, ref["mesh"]), f"{what}: {(m != ref['mesh']).sum()} mesh ids differ"
    assert np.array_equal(tri, ref["triangle"]), f"{what}: {(tri != ref['triangle']).sum()} triangle ids differ"
    assert same_f32(t.view(np.float32), ref["t"]).all(), f"{what}: t differs"


def _check_against_oracle(ctx, crt, ob, flat, rays, dist, torch, traversals=(0, 1), oracle=None):
    """Every ray type, every traversal, against the oracle; returns the oracle's answers for reuse."""
    d_rays = torch.from_numpy(rays).cuda()
    d_dist = torch.from_numpy(dist).cuda()
    oracle = oracle or {}
    for rt in CLOSEST_TYPES + ("RAY_SHADOW",):
        t = getattr(crt, rt)
        if rt not in oracle:
            oracle[rt] = ob.trace_rays(flat, rays, t, dist) if rt == "RAY_SHADOW" else ob.trace_rays(flat, rays, t)
        for trav in traversals:
            if rt == "RAY_SHADOW":
                occ = ctx.trace(d_rays, t, d_dist, traversal=trav).cpu().numpy()
                assert np.array_equal(occ, oracle[rt]), f"{rt} traversal {trav}: {(occ != oracle[rt]).sum()} answers differ"
            else:
                _same_hits(ctx.trace(d_rays, t, traversal=trav), oracle[rt], f"{rt} traversal {trav}")
    return oracle


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_queries_match_oracle(name, gpu, loaded, ob, crt, torch):
    """Every fixture (hw11_room: refractive meshes skipped by shadow queries; many_meshes: the WIDE flavour; empty_scene
    and degenerate_uv: edge cases), every ray type, traversal 0 and 1, and the host wrapper crtb200_trace_rays."""
    sf, flat, _, _ = loaded[name]
    gpu.upload(flat, keepalive=sf)
    rays, dist = caller_rays(flat, 4096, seed=len(name))
    oracle = _check_against_oracle(gpu, crt, ob, flat, rays, dist, torch)
    for trav in (0, 1):
        h, ref = gpu.trace_rays(rays, crt.RAY_PRIMARY, traversal=trav), oracle["RAY_PRIMARY"]
        assert np.array_equal(h["mesh"], ref["mesh"]) and np.array_equal(h["triangle"], ref["triangle"])
        assert same_f32(h["t"], ref["t"]).all()
        assert np.array_equal(gpu.trace_rays(rays, crt.RAY_SHADOW, dist, traversal=trav), oracle["RAY_SHADOW"])
    st = gpu.query_stats()
    assert st["rays_shadow"] == len(rays) and st["rays_primary"] == 0


@pytest.mark.gpu
def test_trees_that_do_not_nest(gpu, handoff, built, scene_dir, ob, crt, torch):
    """A tree whose child boxes stick out of their parent's (as test_trees_that_do_not_nest_take_the_literal_walk
    builds it): queries take the literal walk with no hand-off, even in a context that would hand off every walk."""
    sf = built.SceneFile("hw14_small.crtscene", scene_dir)
    flat = sf.flatten()
    s = flat.contents
    big = max(range(s.n_meshes), key=lambda m: s.meshes[m].n_nodes)
    root = s.mesh_nodes[s.meshes[big].first_node]
    assert root.leaf_count == 0
    root.box_min[0] += 0.25 * (root.box_max[0] - root.box_min[0])
    rays, dist = caller_rays(flat, 4096, seed=5)
    ctx = handoff("all")
    oracle = None
    for c in (gpu, ctx):
        c.upload(flat, keepalive=sf)
        assert not c.debug_scene_layout()["nested_ok"]
        oracle = _check_against_oracle(c, crt, ob, flat, rays, dist, torch, oracle=oracle)
        st = c.query_stats()
        assert st["handoff_closest"] == st["handoff_shadow"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("which", [w for w in HANDOFF if w != "default"])
@pytest.mark.parametrize("name", ["hw14_small", "hw11_room", "many_meshes"])
def test_handoff_settings(name, which, handoff, loaded, ob, crt, torch):
    """Forced, mid-flight, final-pass-only, capped and no hand-off: the same answers; under "all" the k_coop query
    source finished walks of both kinds, under "off" none."""
    ctx = handoff(which)
    sf, flat, _, _ = loaded[name]
    ctx.upload(flat, keepalive=sf)
    rays, dist = caller_rays(flat, 8192, seed=11)
    d_rays, d_dist = torch.from_numpy(rays).cuda(), torch.from_numpy(dist).cuda()
    _same_hits(ctx.trace(d_rays, crt.RAY_PRIMARY), ob.trace_rays(flat, rays, crt.RAY_PRIMARY), which)
    st_c = ctx.query_stats()
    occ = ctx.trace(d_rays, crt.RAY_SHADOW, d_dist).cpu().numpy()
    assert np.array_equal(occ, ob.trace_rays(flat, rays, crt.RAY_SHADOW, dist)), which
    st_s = ctx.query_stats()
    if which == "all":
        assert st_c["handoff_closest"] > 0 and st_s["handoff_shadow"] > 0
    if which == "off":
        assert st_c["handoff_closest"] == 0 and st_s["handoff_shadow"] == 0


@pytest.mark.gpu
def test_several_gpus(gpu, loaded, crt, torch):
    """Context([0, 0, 0]): the batch split into three contiguous ranges gives the single-GPU answers, also for batches
    of 2 and 1 ray (fewer rays than GPUs)."""
    sf, flat, _, _ = loaded["hw14_small"]
    multi = crt.Context([0, 0, 0])
    try:
        for c in (gpu, multi):
            c.upload(flat, keepalive=sf)
        rays, dist = caller_rays(flat, 5000, seed=3)
        d_rays, d_dist = torch.from_numpy(rays).cuda(), torch.from_numpy(dist).cuda()
        for n in (5000, 2, 1):
            for rt in CLOSEST_TYPES:
                t = getattr(crt, rt)
                a, b = gpu.trace(d_rays[:n], t), multi.trace(d_rays[:n], t)
                assert torch.equal(a.records, b.records), (rt, n)
            a = gpu.trace(d_rays[:n], crt.RAY_SHADOW, d_dist[:n])
            b = multi.trace(d_rays[:n], crt.RAY_SHADOW, d_dist[:n])
            assert torch.equal(a, b), n
            assert multi.query_stats()["rays_shadow"] == n
    finally:
        multi.close()


def _light_queries(flat, rays, hits, torch):
    """Shadow queries from the hit points of camera rays to every light: unit directions, max_distance = distance."""
    s = flat.contents
    lights = torch.tensor([list(s.lights[i].position) for i in range(s.n_lights)], dtype=torch.float32, device=rays.device)
    r = rays.reshape(-1, 6)
    hit = hits.mesh.reshape(-1) >= 0
    t = hits.t.reshape(-1).view(torch.float32)[hit]
    p = r[hit, :3] + r[hit, 3:] * t[:, None]
    to = lights[None, :, :] - p[:, None, :]
    dist = torch.linalg.norm(to, dim=2)
    d = to / dist[..., None]
    o = p[:, None, :] + d * 1e-3
    return torch.cat([o, d], dim=2).reshape(-1, 6).contiguous(), dist.reshape(-1).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hw14_dragon_class", "synthetic_10M"])
def test_full_size_camera_and_light_queries(name, gpu, built, crt, torch):
    """Camera rays of hw14_dragon_class at 3840x2160 and synthetic_10M at 1920x1080 from generate_rays_device, traced as
    RAY_PRIMARY, equal the render's primary hits bit for bit; shadow queries from those hits to the lights give the same
    bytes with traversal 0 and 1."""
    bench_mod = importlib.import_module("bench")
    f, folder, kw, tex, depth = bench_mod.ensure_scene(name, {})
    sf = built.SceneFile(f, folder)
    flat = sf.flatten()
    gpu.upload(flat, keepalive=sf)
    cam = sf.camera()
    _, _, ref, _ = gpu.render(cam, crt.make_options(max_depth=depth), want_rgb=False, want_hits=True)
    rays = gpu.generate_rays_device(cam)
    assert tuple(rays.shape) == (sf.info.height, sf.info.width, 6)
    h = gpu.trace(rays, crt.RAY_PRIMARY)
    m = h.mesh.cpu().numpy()
    assert np.array_equal(m, ref["mesh"]) and np.array_equal(h.triangle.cpu().numpy(), ref["triangle"])
    hit = ref["mesh"] >= 0
    assert same_f32(h.t.cpu().numpy().view(np.float32)[hit], ref["t"][hit]).all()
    q, dist = _light_queries(flat, rays, h, torch)
    a = gpu.trace(q, crt.RAY_SHADOW, dist, traversal=0)
    b = gpu.trace(q, crt.RAY_SHADOW, dist, traversal=1)
    assert a.numel() > 0 and torch.equal(a, b)


@pytest.mark.gpu
def test_counting_equals_render(gpu, loaded, crt, torch):
    """count_work = 1: a camera-ray batch of hw14_small (diffuse only) does the render's closest-hit work, test for test."""
    sf, flat, _, _ = loaded["hw14_small"]
    gpu.upload(flat, keepalive=sf)
    cam = sf.camera()
    _, _, _, st = gpu.render(cam, crt.make_options(count_work=1))
    rays = gpu.generate_rays_device(cam)
    gpu.trace(rays, crt.RAY_PRIMARY, count_work=1)
    q = gpu.query_stats()
    assert q["rays_primary"] == rays.shape[0] * rays.shape[1]
    assert q["node_tests_closest"] == st["node_tests_closest"] > 0
    assert q["triangle_tests_closest"] == st["triangle_tests_closest"] > 0
    gpu.trace(rays, crt.RAY_PRIMARY, count_work=2)
    q2 = gpu.query_stats()
    assert 0 < q2["node_tests_closest"] < q["node_tests_closest"]  # culling walks fewer boxes


@pytest.mark.gpu
def test_isolation_and_streams(gpu, loaded, ob, crt, torch):
    """A query between two steps of a progressive session leaves its read equal to the one-shot frame; it leaves
    last_stats(), sampling_stats() and the colour buffer of uncovered pixels alone; and it runs correctly right behind
    a render_device on a non-default stream, with no host synchronisation between them."""
    sf, flat, rects, n = loaded["hw11_room"]
    gpu.upload(flat, keepalive=sf)
    rays, dist = caller_rays(flat, 4096, seed=2)
    d_rays, d_dist = torch.from_numpy(rays).cuda(), torch.from_numpy(dist).cuda()
    cam, opt = sf.camera(), crt.make_options(max_depth=5)
    smp = crt.Sampling.make(gi_samples=1, rays_per_pixel=4, seed=9)
    gpu.set_sampling(smp)
    one, _, _, _ = gpu.render(cam, opt)
    gpu.set_sampling(None)
    p = gpu.progressive(cam, opt, smp)
    p.step(2)
    gpu.trace(d_rays, crt.RAY_PRIMARY)
    gpu.trace(d_rays, crt.RAY_SHADOW, d_dist)
    p.step(2)
    assert same_f32(p.read()[0], one).all()
    p.close()

    sf, flat, rects, n = loaded["uncovered"]
    gpu.upload(flat, keepalive=sf)
    full, _, _, st0 = gpu.render(sf.camera(), crt.make_options())
    ss0 = gpu.sampling_stats()
    last0 = gpu.last_stats()
    gpu.trace(d_rays, crt.RAY_REFLECTION)
    gpu.trace(d_rays, crt.RAY_SHADOW, d_dist)
    assert gpu.query_stats()["rays_shadow"] == len(rays)
    assert gpu.last_stats() == last0 and gpu.sampling_stats() == ss0
    part, _, _, _ = gpu.render(sf.camera(), crt.make_options(rects=rects, n_rects=n))
    assert same_f32(full, part).all()  # the uncovered pixels still hold the full frame

    sf, flat, _, _ = loaded["hw14_small"]
    gpu.upload(flat, keepalive=sf)
    rays, dist = caller_rays(flat, 4096, seed=4)
    want_h = ob.trace_rays(flat, rays, crt.RAY_PRIMARY)
    want_o = ob.trace_rays(flat, rays, crt.RAY_SHADOW, dist)
    s = torch.cuda.Stream()
    frame = torch.empty((sf.info.height, sf.info.width, 3), dtype=torch.float32, device="cuda")
    with torch.cuda.stream(s):
        d_rays, d_dist = torch.from_numpy(rays).cuda(), torch.from_numpy(dist).cuda()
        gpu.render_device(sf.camera(), crt.make_options(), frame.data_ptr(), 0, s.cuda_stream)
        h = gpu.trace(d_rays, crt.RAY_PRIMARY)
        o = gpu.trace(d_rays, crt.RAY_SHADOW, d_dist)
        cam_rays = gpu.generate_rays_device(sf.camera())
    s.synchronize()
    _same_hits(h, want_h, "non-default stream")
    assert np.array_equal(o.cpu().numpy(), want_o)
    assert np.array_equal(cam_rays.cpu().numpy().view(np.uint32), gpu.generate_rays(sf.camera()).view(np.uint32))


def _batch(crt, n, ray_type, rays=0, dist=0, hits=0, occ=0, traversal=0, count_work=0):
    return crt.RayBatch(n=n, ray_type=ray_type, traversal=traversal, count_work=count_work, rays=rays or None,
                        max_distance=dist or None, hits=hits or None, occluded=occ or None)


@pytest.mark.gpu
def test_errors(gpu, loaded, crt, torch):
    sf, flat, _, _ = loaded["hw14_small"]
    gpu.upload(flat, keepalive=sf)
    lib = crt.core()
    n = 64
    rays = torch.zeros((n, 6), dtype=torch.float32, device="cuda")
    rays[:, 5] = -1.0
    dist = torch.ones(n, dtype=torch.float32, device="cuda")
    hits = torch.zeros((n, 3), dtype=torch.int32, device="cuda")
    occ = torch.zeros(n, dtype=torch.uint8, device="cuda")
    raw = torch.zeros(n * 6 + 4, dtype=torch.float32, device="cuda")

    def rc(b):
        return lib.crtb200_trace_rays_device(gpu._h, C.byref(b), None)

    assert rc(_batch(crt, n, crt.RAY_PRIMARY, rays.data_ptr(), hits=hits.data_ptr())) == 0
    assert rc(_batch(crt, n, crt.RAY_SHADOW, rays.data_ptr(), dist.data_ptr(), occ=occ.data_ptr())) == 0
    torch.cuda.synchronize()
    # host memory
    h_rays = np.zeros((n, 6), np.float32)
    h_hits = np.zeros((n, 3), np.int32)
    assert rc(_batch(crt, n, crt.RAY_PRIMARY, h_rays.ctypes.data, hits=hits.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, crt.RAY_PRIMARY, rays.data_ptr(), hits=h_hits.ctypes.data)) == ERR_ARG
    # misalignment
    assert rc(_batch(crt, n, crt.RAY_PRIMARY, raw.data_ptr() + 2, hits=hits.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, crt.RAY_SHADOW, rays.data_ptr(), dist.data_ptr() + 1, occ=occ.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, crt.RAY_PRIMARY, raw.data_ptr() + 4, hits=hits.data_ptr())) == 0  # 4-byte aligned is enough
    # ray types, missing outputs, modes, sizes
    assert rc(_batch(crt, n, crt.RAY_DIFFUSE, rays.data_ptr(), hits=hits.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, crt.RAY_PRIMARY, rays.data_ptr(), occ=occ.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, crt.RAY_SHADOW, rays.data_ptr(), occ=occ.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, crt.RAY_SHADOW, rays.data_ptr(), dist.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, crt.RAY_PRIMARY, rays.data_ptr(), hits=hits.data_ptr(), traversal=2)) == ERR_ARG
    assert rc(_batch(crt, n, crt.RAY_PRIMARY, rays.data_ptr(), hits=hits.data_ptr(), count_work=3)) == ERR_ARG
    assert rc(_batch(crt, 1 << 31, crt.RAY_PRIMARY, rays.data_ptr(), hits=hits.data_ptr())) == ERR_ARG
    # n = 0: nothing to do, nothing written
    hits.fill_(7)
    assert rc(_batch(crt, 0, crt.RAY_PRIMARY, rays.data_ptr(), hits=hits.data_ptr())) == 0
    torch.cuda.synchronize()
    assert int(hits.min()) == 7 == int(hits.max())
    assert gpu.trace(rays[:0], crt.RAY_PRIMARY).mesh.shape == (0,)
    # another device's memory
    if torch.cuda.device_count() > 1:
        other = torch.zeros((n, 6), dtype=torch.float32, device="cuda:1")
        assert rc(_batch(crt, n, crt.RAY_PRIMARY, other.data_ptr(), hits=hits.data_ptr())) == ERR_ARG
    # the Python layer refuses wrong dtype, device and shape before the C call
    for bad in (rays.double(), rays.cpu(), rays[:, :5], rays.reshape(-1)):
        with pytest.raises(crt.CrtError):
            gpu.trace(bad, crt.RAY_PRIMARY)
    with pytest.raises(crt.CrtError):
        gpu.trace(rays, crt.RAY_SHADOW)  # no max_distance
    with pytest.raises(crt.CrtError):
        gpu.trace(rays, crt.RAY_SHADOW, dist[:-1])
    with pytest.raises(crt.CrtError):
        gpu.trace(rays, crt.RAY_DIFFUSE)
    with pytest.raises(crt.CrtError):
        gpu.trace(rays, crt.RAY_PRIMARY, out=torch.zeros((n, 3), dtype=torch.float32, device="cuda"))
    # out= reuses the caller's buffer
    h = gpu.trace(rays, crt.RAY_PRIMARY, out=hits)
    assert h.mesh.data_ptr() == hits.data_ptr()
    assert gpu.trace(rays, crt.RAY_PRIMARY, out=h).records is hits
    # ... also when that buffer is itself a view of a larger tensor
    big = torch.zeros((2 * n, 3), dtype=torch.int32, device="cuda")
    h = gpu.trace(rays, crt.RAY_PRIMARY, out=big[n:])
    h2 = gpu.trace(rays, crt.RAY_PRIMARY, out=h)
    assert h2.records.data_ptr() == big[n:].data_ptr() and torch.equal(big[n:], hits)
    # 2^31 rays or more are refused before anything is copied or traced
    with pytest.raises(crt.CrtError, match="2\\^31"):
        gpu.trace(rays[:1].expand(1 << 31, 6), crt.RAY_PRIMARY)
    assert gpu.trace(rays, crt.RAY_SHADOW, dist, out=occ).data_ptr() == occ.data_ptr()
    # device camera rays: host or misaligned destinations
    assert lib.crtb200_generate_rays_device(gpu._h, C.byref(sf.camera()), h_rays.ctypes.data, None) == ERR_ARG
    assert lib.crtb200_generate_rays_device(gpu._h, C.byref(sf.camera()), raw.data_ptr() + 2, None) == ERR_ARG
    # no scene
    fresh = crt.Context(0)
    try:
        assert lib.crtb200_trace_rays_device(fresh._h, C.byref(_batch(crt, n, crt.RAY_PRIMARY, rays.data_ptr(), hits=hits.data_ptr())), None) == ERR_STATE
        assert lib.crtb200_generate_rays_device(fresh._h, C.byref(sf.camera()), rays.data_ptr(), None) == ERR_STATE
        with pytest.raises(crt.CrtError, match="no scene"):
            fresh.generate_rays_device(sf.camera())
    finally:
        fresh.close()


# ---- no GPU needed ----------------------------------------------------------------------------------------------
def test_abi_exports_and_null_context(built):
    lib = built.core()
    for name in ("crtb200_trace_rays_device", "crtb200_generate_rays_device", "crtb200_last_query_stats"):
        assert hasattr(lib, name)
    b = built.RayBatch(n=1, ray_type=built.RAY_PRIMARY)
    assert lib.crtb200_trace_rays_device(None, C.byref(b), None) == ERR_ARG
    assert lib.crtb200_generate_rays_device(None, C.byref(built.Camera.make()), None, None) == ERR_ARG
    assert lib.crtb200_last_query_stats(None, C.byref(built.Stats())) == ERR_ARG


def test_ray_batch_layout_matches_header(built, tmp_path):
    """The ctypes RayBatch against the C compiler's layout of crtb200_ray_batch."""
    src = tmp_path / "layout.c"
    fields = [f for f, _ in built.RayBatch._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "crtb200.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(crtb200_ray_batch));\n' +
                   "".join(f'  printf(" %zu", offsetof(crtb200_ray_batch, {f}));\n' for f in fields) + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [C.sizeof(built.RayBatch)] + [getattr(built.RayBatch, f).offset for f in fields]
