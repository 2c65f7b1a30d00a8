"""Caller-supplied rays shaded on the GPU (crtb200_shade_rays_device, Context.shade; DESIGN.md 3.13): colour i is
RayTracer::shootRay(ray i, 0) bit for bit -- the CPU oracle's shoot_ray, or shoot_gi under the sampling contract --
through the frame pipeline, for any direction length and ray type, under every hand-off setting, on several GPUs, on
non-default streams and in chunks, without touching the context's frame state.  Shading the camera rays of a frame
gives the frame.  The last tests need no GPU: the C ABI surface and the oracle's own identities."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

import shade_oracle as so
from conftest import ROOT, SMALL_SCENES, frame_digests, same_f32
from gi_oracle import HIT_DTYPE, render_sampled
from handoff_contexts import HANDOFF, HandoffContexts
from test_gpu_ray_queries import caller_rays

ERR_ARG, ERR_STATE = -1, -3
SHADE_TYPES = ("RAY_PRIMARY", "RAY_REFLECTION", "RAY_REFRACTION")
RAY_KEYS = ("rays_primary", "rays_shadow", "rays_reflection", "rays_refraction")


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


def _hits_np(h):
    return np.ascontiguousarray(h.records.cpu().numpy()).view(HIT_DTYPE)[..., 0]


def _same(rgb, hits, ref_rgb, ref_hits, what):
    got = rgb.cpu().numpy().reshape(-1, 3)
    same = same_f32(got, np.asarray(ref_rgb).reshape(-1, 3))
    assert same.all(), f"{what}: {(~same).any(axis=1).sum()} colours differ"
    if hits is not None:
        h, r = _hits_np(hits).reshape(-1), np.asarray(ref_hits).reshape(-1)
        assert np.array_equal(h["mesh"], r["mesh"]) and np.array_equal(h["triangle"], r["triangle"]), f"{what}: hit ids differ"
        assert same_f32(h["t"], r["t"]).all(), f"{what}: hit t differs"


def _rays_of(st):
    return [st[k] for k in RAY_KEYS]


def _shade_vs_oracle(ctx, crt, flat, rays, d_rays, rt, depth, traversal, count_work=0, what=""):
    opt = crt.make_options(max_depth=depth)
    ref_rgb, ref_hits, ref_st = so.shade_rays(flat, rays, rt, opt)
    rgb, h = ctx.shade(d_rays, rt, max_depth=depth, traversal=traversal, count_work=count_work, want_hits=True)
    _same(rgb, h, ref_rgb, ref_hits, what)
    st = ctx.last_stats()
    assert _rays_of(st) == _rays_of(ref_st), what
    if count_work == 1:
        for k in ("node_tests_closest", "triangle_tests_closest", "node_tests_shadow", "triangle_tests_shadow"):
            assert st[k] == ref_st[k], (what, k)
    return st


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_shade_matches_oracle(name, gpu, loaded, crt, torch):
    """Every fixture, every ray type, max_depth 0 / 1 / 5, traversal 0 / 1: colours, hits and ray counts as the oracle's
    shoot_ray; with count_work = 1 the node and triangle tests too."""
    sf, flat, _, _ = loaded[name]
    gpu.upload(flat, keepalive=sf)
    rays, _ = caller_rays(flat, 2048, seed=len(name) + 1)
    d_rays = torch.from_numpy(rays).cuda()
    for rt in SHADE_TYPES:
        t = getattr(crt, rt)
        for depth in (0, 1, 5):
            for trav in (0, 1):
                _shade_vs_oracle(gpu, crt, flat, rays, d_rays, t, depth, trav, what=f"{name} {rt} depth {depth} traversal {trav}")
        _shade_vs_oracle(gpu, crt, flat, rays, d_rays, t, 5, 0, count_work=1, what=f"{name} {rt} count_work 1")


@pytest.mark.gpu
def test_trees_that_do_not_nest(gpu, handoff, built, scene_dir, crt, torch):
    """A tree whose child boxes stick out of their parent's (built as the query test builds it): the literal walk, no
    hand-off, the oracle's colours -- also in a context that would hand off every walk."""
    sf = built.SceneFile("hw14_small.crtscene", scene_dir)
    flat = sf.flatten()
    s = flat.contents
    big = max(range(s.n_meshes), key=lambda m: s.meshes[m].n_nodes)
    root = s.mesh_nodes[s.meshes[big].first_node]
    assert root.leaf_count == 0
    root.box_min[0] += 0.25 * (root.box_max[0] - root.box_min[0])
    rays, _ = caller_rays(flat, 4096, seed=5)
    d_rays = torch.from_numpy(rays).cuda()
    for c in (gpu, handoff("all")):
        c.upload(flat, keepalive=sf)
        assert not c.debug_scene_layout()["nested_ok"]
        for rt in SHADE_TYPES:
            st = _shade_vs_oracle(c, crt, flat, rays, d_rays, getattr(crt, rt), 5, 0, what=rt)
            assert st["handoff_closest"] == st["handoff_shadow"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_camera_rays_give_the_frame(name, gpu, loaded, crt, torch):
    """The once-normalised getRay ray of every pixel, shaded as RAY_PRIMARY, gives render()'s colours, hits and ray
    counts."""
    sf, flat, _, _ = loaded[name]
    gpu.upload(flat, keepalive=sf)
    cam, opt = sf.camera(), crt.make_options(max_depth=5)
    rgb, _, hits, st = gpu.render(cam, opt, want_hits=True)
    rays = torch.from_numpy(so.camera_rays(flat, cam)).cuda()
    got, h = gpu.shade(rays, crt.RAY_PRIMARY, max_depth=5, want_hits=True)
    assert tuple(got.shape) == rgb.shape
    _same(got, h, rgb, hits, name)
    assert _rays_of(gpu.last_stats()) == _rays_of(st)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hw11_room", "hw14_dragon_class"])
def test_full_size_camera_rays(name, gpu, built, ob, crt, torch):
    """hw11_room at 1920x1080 and hw14_dragon_class at 3840x2160: the shaded camera rays against the stored frames'
    digests (float RGB, PPM bytes quantised on the host, hits) and ray counts."""
    bench_mod = importlib.import_module("bench")
    f, folder, kw, tex, depth = bench_mod.ensure_scene(name, {})
    ref = np.load(os.path.join(ROOT, "tests", "golden", "fullsize_" + name + ".npz"))
    sf = built.SceneFile(f, folder)
    flat = sf.flatten()
    gpu.upload(flat, keepalive=sf)
    cam = sf.camera()
    assert np.array_equal(np.array(list(cam.position) + list(cam.rotation), np.float32), ref["camera"])
    rays = torch.from_numpy(so.camera_rays(flat, cam)).cuda()
    rgb, h = gpu.shade(rays, crt.RAY_PRIMARY, max_depth=depth, want_hits=True)
    st = gpu.last_stats()
    rgb = rgb.cpu().numpy()
    for k, v in frame_digests(rgb, ob.quantize(rgb), _hits_np(h)).items():
        assert v == str(ref[k + "_sha256"]), k
    assert _rays_of(st) == list(ref["rays"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hw11_room", "hw12_textures", "hw14_small"])
def test_gi_matches_oracle(name, gpu, loaded, crt, torch):
    """GI on: G = 1, 2, 4 at max_depth 2-5, every ray type, a sample word and first index of their own: colours, hits,
    ray counts and diffuse rays as the oracle's shoot_gi."""
    sf, flat, _, _ = loaded[name]
    gpu.upload(flat, keepalive=sf)
    rays, _ = caller_rays(flat, 512, seed=7)
    d_rays = torch.from_numpy(rays).cuda()
    try:
        for g in (1, 2, 4):
            smp = crt.Sampling.make(gi_samples=g, rays_per_pixel=3, seed=21 + g, frame_index=2)
            gpu.set_sampling(smp)
            for depth in (2, 3, 4, 5):
                rt = getattr(crt, SHADE_TYPES[depth % 3])
                sample, first = 5 + depth, (1 << 32) - 100 if depth == 4 else 1000 * depth
                opt = crt.make_options(max_depth=depth)
                ref_rgb, ref_hits, ref_st = so.shade_rays(flat, rays, rt, opt, smp, sample, first)
                rgb, h = gpu.shade(d_rays, rt, max_depth=depth, sample=sample, first_index=first, want_hits=True)
                what = f"{name} G {g} depth {depth}"
                _same(rgb, h, ref_rgb, ref_hits, what)
                assert _rays_of(gpu.last_stats()) == _rays_of(ref_st), what
                assert gpu.sampling_stats() == {"rays_diffuse": ref_st["rays_diffuse"], "samples": 1}, what
    finally:
        gpu.set_sampling(None)


@pytest.mark.gpu
def test_gi_samples_give_the_frame(gpu, loaded, crt, torch):
    """Jittered camera rays of sample 0 give the rays_per_pixel = 1 GI frame; samples 0..3 summed in order and divided
    by 4 give the rays_per_pixel = 4 frame; a batch shaded as two calls (first_index 0 and k) equals one call."""
    sf, flat, _, _ = loaded["hw11_room"]
    gpu.upload(flat, keepalive=sf)
    cam, opt = sf.camera(), crt.make_options(max_depth=4)
    h, w = sf.info.height, sf.info.width
    try:
        for rpp in (1, 4):
            smp = crt.Sampling.make(gi_samples=2, rays_per_pixel=rpp, seed=3)
            gpu.set_sampling(smp)
            frame, _, _, _ = gpu.render(cam, opt)
            acc = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
            for s in range(rpp):
                rays = torch.from_numpy(so.camera_rays(flat, cam, smp, s)).cuda()
                rgb, _ = gpu.shade(rays, crt.RAY_PRIMARY, max_depth=4, sample=s)
                acc = acc + rgb
            _same(acc / float(rpp), None, frame, None, f"rays_per_pixel {rpp}")
        rays = torch.from_numpy(so.camera_rays(flat, cam, smp, 2)).cuda().reshape(-1, 6)
        one, _ = gpu.shade(rays, crt.RAY_PRIMARY, max_depth=4, sample=2)
        k = 5003
        a, _ = gpu.shade(rays[:k], crt.RAY_PRIMARY, max_depth=4, sample=2, first_index=0)
        b, _ = gpu.shade(rays[k:], crt.RAY_PRIMARY, max_depth=4, sample=2, first_index=k)
        assert torch.equal(torch.cat([a, b]).view(torch.int32), one.view(torch.int32))
    finally:
        gpu.set_sampling(None)


@pytest.mark.gpu
@pytest.mark.parametrize("which", [w for w in HANDOFF if w != "default"])
@pytest.mark.parametrize("name", ["hw14_small", "hw11_room", "many_meshes"])
def test_handoff_settings(name, which, handoff, loaded, crt, torch):
    """Forced, mid-flight, final-pass-only, capped and no hand-off: the oracle's colours; under "all" the level-0
    walks went through k_coop over the caller's rays (ShadeRays), under "off" nothing was handed off."""
    ctx = handoff(which)
    sf, flat, _, _ = loaded[name]
    ctx.upload(flat, keepalive=sf)
    rays, _ = caller_rays(flat, 4096, seed=11)
    d_rays = torch.from_numpy(rays).cuda()
    for rt in ("RAY_PRIMARY", "RAY_REFLECTION"):
        st = _shade_vs_oracle(ctx, crt, flat, rays, d_rays, getattr(crt, rt), 5, 0, what=f"{which} {rt}")
        if which == "all":
            assert st["handoff_closest"] > 0
        if which == "off":
            assert st["handoff_closest"] == st["handoff_shadow"] == 0


@pytest.mark.gpu
def test_several_gpus_and_streams(gpu, loaded, crt, torch):
    """The same colours and hits on a [0, 0, 0] context (also for 2 and 1 rays) and on a non-default stream right behind
    a render_device; GI batches keep their pixel index across the GPUs' ranges."""
    sf, flat, _, _ = loaded["hw14_small"]
    gpu.upload(flat, keepalive=sf)
    rays, _ = caller_rays(flat, 12288, seed=3)
    d_rays = torch.from_numpy(rays).cuda()
    ref_rgb, ref_hits, _ = so.shade_rays(flat, rays, crt.RAY_REFLECTION, crt.make_options(max_depth=5))
    multi = crt.Context([0, 0, 0])
    try:
        multi.upload(flat, keepalive=sf)
        for n in (12288, 2, 1):
            rgb, h = multi.shade(d_rays[:n], crt.RAY_REFLECTION, want_hits=True)
            _same(rgb, h, ref_rgb[:n], ref_hits[:n], f"3 GPUs, {n} rays")
        assert _rays_of(multi.last_stats()) == _rays_of(so.shade_rays(flat, rays[:1], crt.RAY_REFLECTION, crt.make_options())[2])
        smp = crt.Sampling.make(gi_samples=2, seed=4)
        for c in (gpu, multi):
            c.set_sampling(smp)
        a, _ = gpu.shade(d_rays, crt.RAY_PRIMARY, sample=1, first_index=77)
        b, _ = multi.shade(d_rays, crt.RAY_PRIMARY, sample=1, first_index=77)
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    finally:
        gpu.set_sampling(None)
        multi.close()

    s = torch.cuda.Stream()
    frame = torch.empty((sf.info.height, sf.info.width, 3), dtype=torch.float32, device="cuda")
    with torch.cuda.stream(s):
        d2 = torch.from_numpy(rays).cuda()
        gpu.render_device(sf.camera(), crt.make_options(), frame.data_ptr(), 0, s.cuda_stream)
        rgb, h = gpu.shade(d2, crt.RAY_REFLECTION, want_hits=True)
    s.synchronize()
    _same(rgb, h, ref_rgb, ref_hits, "non-default stream")


@pytest.mark.gpu
def test_queue_budget_chunks(gpu, loaded, crt, torch):
    """The smallest queue budget (64 MiB) splits 30 000 rays of hw11_room at depth 5 (ray trees of up to 63 nodes)
    into at least three chunks -- kernel_launches grows with them -- and changes no colour, hit or count."""
    sf, flat, _, _ = loaded["hw11_room"]
    gpu.upload(flat, keepalive=sf)
    rays, _ = caller_rays(flat, 30000, seed=8)
    d_rays = torch.from_numpy(rays).cuda()
    a, ha = gpu.shade(d_rays, crt.RAY_REFLECTION, want_hits=True)
    st_a = gpu.last_stats()
    gpu.set_queue_budget(64 << 20)
    try:
        b, hb = gpu.shade(d_rays, crt.RAY_REFLECTION, want_hits=True)
        st_b = gpu.last_stats()
    finally:
        gpu.set_queue_budget(16 << 30)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32)) and torch.equal(ha.records, hb.records)
    assert st_b["kernel_launches"] >= 3 * st_a["kernel_launches"]
    assert _rays_of(st_a) == _rays_of(st_b)


@pytest.mark.gpu
def test_isolation(gpu, loaded, crt, torch):
    """A shade call between two progressive steps leaves the session's read equal to the one-shot frame; a partial
    render after it keeps the earlier uncovered pixels; query_stats() is unchanged; a render after a shade with another
    max_depth equals a fresh context's."""
    sf, flat, rects, n = loaded["hw11_room"]
    gpu.upload(flat, keepalive=sf)
    rays, _ = caller_rays(flat, 4096, seed=2)
    d_rays = torch.from_numpy(rays).cuda()
    cam, opt = sf.camera(), crt.make_options(max_depth=5)
    smp = crt.Sampling.make(gi_samples=1, rays_per_pixel=4, seed=9)
    gpu.set_sampling(smp)
    one, _, _, _ = gpu.render(cam, opt)
    gpu.set_sampling(None)
    p = gpu.progressive(cam, opt, smp)
    p.step(2)
    gpu.shade(d_rays, crt.RAY_PRIMARY, max_depth=2)
    p.step(2)
    assert same_f32(p.read()[0], one).all()
    p.close()

    gpu.trace(d_rays, crt.RAY_PRIMARY)
    q0 = gpu.query_stats()
    sf, flat, rects, n = loaded["uncovered"]
    gpu.upload(flat, keepalive=sf)
    full, _, _, _ = gpu.render(sf.camera(), crt.make_options())
    gpu.shade(d_rays, crt.RAY_REFRACTION, max_depth=3)
    torch.cuda.synchronize()
    assert gpu.query_stats() == q0
    part, _, _, _ = gpu.render(sf.camera(), crt.make_options(rects=rects, n_rects=n))
    assert same_f32(full, part).all()  # the uncovered pixels still hold the full frame

    sf, flat, _, _ = loaded["hw07_scene0b"]
    gpu.upload(flat, keepalive=sf)
    gpu.shade(d_rays, crt.RAY_PRIMARY, max_depth=1)
    torch.cuda.synchronize()  # (the shade ran on torch's stream, the render runs on the context's own)
    after, _, _, st = gpu.render(sf.camera(), crt.make_options(max_depth=5))
    fresh = crt.Context(0)
    try:
        fresh.upload(flat, keepalive=sf)
        ref, _, _, st_ref = fresh.render(sf.camera(), crt.make_options(max_depth=5))
    finally:
        fresh.close()
    assert same_f32(after, ref).all() and _rays_of(st) == _rays_of(st_ref)


def _batch(crt, n, ray_type, rays=0, rgb=0, hits=0, traversal=0, count_work=0, max_depth=5):
    return crt.ShadeBatch(n=n, ray_type=ray_type, traversal=traversal, count_work=count_work, max_depth=max_depth,
                          rays=rays or None, rgb=rgb or None, hits=hits or None)


@pytest.mark.gpu
def test_errors(gpu, loaded, crt, torch):
    sf, flat, _, _ = loaded["hw14_small"]
    gpu.upload(flat, keepalive=sf)
    lib = crt.core()
    n = 64
    rays = torch.zeros((n, 6), dtype=torch.float32, device="cuda")
    rays[:, 5] = -1.0
    rgb = torch.zeros((n, 3), dtype=torch.float32, device="cuda")
    hits = torch.zeros((n, 3), dtype=torch.int32, device="cuda")
    raw = torch.zeros(n * 6 + 4, dtype=torch.float32, device="cuda")

    def rc(b, ctx=gpu):
        return lib.crtb200_shade_rays_device(ctx._h, C.byref(b) if b is not None else None, None)

    P = crt.RAY_PRIMARY
    assert rc(_batch(crt, n, P, rays.data_ptr(), rgb.data_ptr(), hits.data_ptr())) == 0
    assert rc(_batch(crt, n, P, rays.data_ptr(), rgb.data_ptr())) == 0  # hits are optional
    torch.cuda.synchronize()
    assert rc(None) == ERR_ARG
    assert rc(_batch(crt, n, P, 0, rgb.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, P, rays.data_ptr(), 0)) == ERR_ARG
    h_rays, h_rgb, h_hits = np.zeros((n, 6), np.float32), np.zeros((n, 3), np.float32), np.zeros((n, 3), np.int32)
    assert rc(_batch(crt, n, P, h_rays.ctypes.data, rgb.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, P, rays.data_ptr(), h_rgb.ctypes.data)) == ERR_ARG
    assert rc(_batch(crt, n, P, rays.data_ptr(), rgb.data_ptr(), h_hits.ctypes.data)) == ERR_ARG
    assert rc(_batch(crt, n, P, raw.data_ptr() + 2, rgb.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, P, rays.data_ptr(), rgb.data_ptr() + 1)) == ERR_ARG
    assert rc(_batch(crt, n, P, rays.data_ptr(), rgb.data_ptr(), hits.data_ptr() + 2)) == ERR_ARG
    assert rc(_batch(crt, n, P, raw.data_ptr() + 4, rgb.data_ptr())) == 0  # 4-byte aligned is enough
    for t in (crt.RAY_SHADOW, crt.RAY_DIFFUSE, 7):
        assert rc(_batch(crt, n, t, rays.data_ptr(), rgb.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, P, rays.data_ptr(), rgb.data_ptr(), traversal=2)) == ERR_ARG
    assert rc(_batch(crt, n, P, rays.data_ptr(), rgb.data_ptr(), count_work=3)) == ERR_ARG
    assert rc(_batch(crt, n, P, rays.data_ptr(), rgb.data_ptr(), max_depth=32)) == ERR_ARG
    assert rc(_batch(crt, 1 << 31, P, rays.data_ptr(), rgb.data_ptr())) == ERR_ARG
    assert rc(_batch(crt, n, P, rays.data_ptr(), rgb.data_ptr(), max_depth=31)) == 0
    torch.cuda.synchronize()
    # n = 0: nothing to do, nothing written
    rgb.fill_(7)
    assert rc(_batch(crt, 0, P, rays.data_ptr(), rgb.data_ptr())) == 0
    torch.cuda.synchronize()
    assert float(rgb.min()) == 7.0 == float(rgb.max())
    assert gpu.shade(rays[:0])[0].shape == (0, 3)
    if torch.cuda.device_count() > 1:
        other = torch.zeros((n, 6), dtype=torch.float32, device="cuda:1")
        assert rc(_batch(crt, n, P, other.data_ptr(), rgb.data_ptr())) == ERR_ARG
    # the Python layer refuses wrong dtype, device, shape and ray type before the C call
    for bad in (rays.double(), rays.cpu(), rays[:, :5], rays.reshape(-1)):
        with pytest.raises(crt.CrtError):
            gpu.shade(bad)
    for t in (crt.RAY_SHADOW, crt.RAY_DIFFUSE):
        with pytest.raises(crt.CrtError):
            gpu.shade(rays, t)
    for bad_out in (torch.zeros((n, 3), dtype=torch.float64, device="cuda"), torch.zeros((n, 4), dtype=torch.float32, device="cuda"),
                    torch.zeros((3, n), dtype=torch.float32, device="cuda").t()):
        with pytest.raises(crt.CrtError):
            gpu.shade(rays, out=bad_out)
    with pytest.raises(crt.CrtError):
        gpu.shade(rays, max_depth=32)
    with pytest.raises(crt.CrtError, match="2\\^31"):
        gpu.shade(rays[:1].expand(1 << 31, 6))
    got, h = gpu.shade(rays, out=rgb, want_hits=True)
    assert got.data_ptr() == rgb.data_ptr() and h.records.shape == (n, 3)
    fresh = crt.Context(0)
    try:
        assert rc(_batch(crt, n, P, rays.data_ptr(), rgb.data_ptr()), fresh) == ERR_STATE
        with pytest.raises(crt.CrtError, match="no scene"):
            fresh.shade(rays)
    finally:
        fresh.close()


# ---- no GPU needed ----------------------------------------------------------------------------------------------
def test_abi_export_and_null_context(built):
    lib = built.core()
    assert hasattr(lib, "crtb200_shade_rays_device")
    b = built.ShadeBatch(n=1, ray_type=built.RAY_PRIMARY)
    assert lib.crtb200_shade_rays_device(None, C.byref(b), None) == ERR_ARG


def test_shade_batch_layout_matches_header(built, tmp_path):
    """The ctypes ShadeBatch against the C compiler's layout of crtb200_shade_batch."""
    src = tmp_path / "layout.c"
    fields = [f for f, _ in built.ShadeBatch._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "crtb200.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(crtb200_shade_batch));\n' +
                   "".join(f'  printf(" %zu", offsetof(crtb200_shade_batch, {f}));\n' for f in fields) + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [C.sizeof(built.ShadeBatch)] + [getattr(built.ShadeBatch, f).offset for f in fields]


@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_oracle_camera_rays_give_the_frame(name, loaded, ob, crt):
    """The oracle's own identities: shade_rays of the camera rays is crt_oracle_render's frame and ray counts; the
    sampled variant over samples 0..N-1, summed in order and divided by N, is crt_oracle_render_sampled's frame at
    rays_per_pixel 1 and 4 (hits: sample 0's)."""
    sf, flat, _, _ = loaded[name]
    cam, opt = sf.camera(), crt.make_options(max_depth=5)
    h, w = sf.info.height, sf.info.width
    rgb, hits, st = ob.render(flat, cam, opt)
    got, got_hits, got_st = so.shade_rays(flat, so.camera_rays(flat, cam), crt.RAY_PRIMARY, opt)
    assert same_f32(got.reshape(h, w, 3), rgb).all()
    hits = hits.reshape(-1)
    assert np.array_equal(got_hits["mesh"], hits["mesh"]) and np.array_equal(got_hits["triangle"], hits["triangle"])
    assert same_f32(got_hits["t"], hits["t"]).all()
    assert _rays_of(got_st) == _rays_of(st)
    opt = crt.make_options(max_depth=3)
    for rpp in (1, 4):
        smp = crt.Sampling.make(gi_samples=2, rays_per_pixel=rpp, seed=13)
        ref, ref_hits, ref_st = render_sampled(flat, cam, opt, smp)
        acc = np.zeros((h * w, 3), np.float32)
        diffuse = 0
        for s in range(rpp):
            c, hs, st_s = so.shade_rays(flat, so.camera_rays(flat, cam, smp, s), crt.RAY_PRIMARY, opt, smp, s, 0)
            acc = acc + c
            diffuse += st_s["rays_diffuse"]
            if s == 0:
                assert np.array_equal(hs["mesh"], ref_hits["mesh"].reshape(-1))
        assert same_f32((acc / np.float32(rpp)).reshape(h, w, 3), ref).all(), rpp
        assert diffuse == ref_st["rays_diffuse"]
