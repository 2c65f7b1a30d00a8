"""GPU: crtb200_update_vertices_device / Context.update_vertices (DESIGN.md 3.14).  After an update the context must hold
exactly what crtb200_upload_geometry leaves for the scene with the new positions and Mesh::Mesh's normals of them
(tests/update_oracle.py): layout, triangle records, vertex normals, trees, and so every frame, query and shade."""
import ctypes as C

import numpy as np
import pytest

import kd_build_oracle as kb
import shade_oracle as so
import update_oracle as uo
from conftest import SMALL_SCENES, same_f32
from test_gpu_device_build import _assert_frames_equal, _frames, assert_layout_equal
from test_gpu_fullsize import _load
from test_gpu_parity import _covered
from test_gpu_ray_queries import caller_rays

pytestmark = pytest.mark.gpu
ERR_ARG, ERR_STATE = -1, -3
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
def ref_ctx(built):
    ctx = built.Context(0)
    yield ctx
    ctx.close()


def _state(ctx, d=0):
    geom, vn = ctx.debug_scene_geometry(d)
    return ctx.debug_scene_layout(d), geom, vn


def _assert_state_equal(a, b):
    assert_layout_equal(a[0], b[0])
    assert a[1].shape == b[1].shape and same_f32(a[1], b[1]).all(), "triangle records differ"
    assert a[2].shape == b[2].shape and same_f32(a[2], b[2]).all(), "vertex normals differ"


def _trees(ctx):
    return kb.device_trees(ctx.scene_trees())


def _mesh_vertices(flat):
    """Per mesh the sorted global ids of the vertices its triangles use."""
    a = kb.scene_arrays(flat)
    tv, m = a["triangle_vertex"], a["meshes"]
    return [np.unique(tv[f:f + n]) for f, n in zip(m["first_triangle"].tolist(), m["n_triangles"].tolist())]


def _largest_meshes(flat):
    verts = _mesh_vertices(flat)
    return sorted(range(len(verts)), key=lambda i: -len(verts[i]))


def _deform(vp, amp=0.05, phase=0.0):
    """A smooth displacement of every vertex (the sphere-style deformation of the tests), in float32."""
    with np.errstate(all="ignore"):
        s = np.sin(np.float32(3.0) * vp[:, 0] + np.float32(2.0) * vp[:, 1] + np.float32(phase)).astype(np.float32)
        return (vp * (np.float32(1.0) + np.float32(amp) * s)[:, None]).astype(np.float32)


def _edits(flat):
    """(name, positions) of the edits every fixture goes through."""
    vp = kb.scene_arrays(flat)["vertex_position"]
    if len(vp) == 0:
        return []
    order = _largest_meshes(flat)
    verts = _mesh_vertices(flat)
    out = []
    p = vp.copy()
    p[verts[order[0]]] += np.array([0.3, -0.2, 0.15], np.float32)
    out.append(("rigid", p))
    p = vp.copy()
    tgt = order[1] if len(order) > 1 else order[0]
    # scaled towards the origin by 1e-25: every cross product underflows, so every face normal of the mesh is zero, while
    # the boxes keep their order (a true point would put every triangle on both sides of every split: 2^25 nodes)
    p[verts[tgt]] *= np.float32(1e-25)
    out.append(("to_point", p))
    p = vp.copy()
    z = p == 0
    p[z] = np.where(np.signbit(p[z]), np.float32(0.0), np.float32(-0.0))  # every zero flips its sign
    p[::2] = p[::2] + np.float32(-0.0)  # -0.0 shifts: x + -0 = x, -0 + -0 = -0
    v = verts[order[0]]
    p[v[:64]] = np.round(p[v[:64]] * 64) / 64  # ties: small moves onto a 1/64 grid (shared box bounds, split positions)
    out.append(("signed_zero_ties", p))
    # (+inf only: a -inf bound makes the split planes NaN, and then every split keeps every element on both sides)
    p = vp.copy()
    p[verts[order[0]][0]] = [np.nan, np.inf, 0.5]
    p[verts[order[-1]][-1]] = [np.inf, np.nan, np.inf]
    out.append(("nan_inf", p))
    out.append(("deform", _deform(vp)))
    return out


def _update(ctx, torch, positions):
    ctx.update_vertices(torch.from_numpy(np.ascontiguousarray(positions, np.float32)).cuda())


@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_identity_update(name, gpu, loaded, built, torch):
    """3: updating with the uploaded positions changes nothing, after upload_scene and after upload_geometry."""
    sf, flat, _, _ = loaded[name]
    vp = built.scene_vertex_positions(flat)
    gpu.upload(flat, keepalive=sf)
    before = _state(gpu)
    _update(gpu, torch, vp)
    _assert_state_equal(_state(gpu), before)
    kb.assert_trees_equal(_trees(gpu), kb.host_trees(flat))
    gpu.upload_geometry(sf.flatten(trees=False), keepalive=sf)
    before, trees = _state(gpu), _trees(gpu)
    _update(gpu, torch, vp)
    _assert_state_equal(_state(gpu), before)
    kb.assert_trees_equal(_trees(gpu), trees)


@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_edited_geometry(name, gpu, ref_ctx, loaded, built, ob, torch):
    """4: every edit equals upload_geometry of the edited copy: state, trees, frames and counters; the deformed scene's
    unsampled frame equals the CPU oracle's."""
    sf, flat, rects, n = loaded[name]
    for i, (edit, p) in enumerate(_edits(flat)):
        if i % 2:
            gpu.upload(flat, keepalive=sf)
        else:
            gpu.upload_geometry(sf.flatten(trees=False), keepalive=sf)
        _update(gpu, torch, p)
        e = uo.EditedScene(built, flat, p)
        ref_ctx.upload_geometry(e.ptr, keepalive=e)
        _assert_state_equal(_state(gpu), _state(ref_ctx))
        kb.assert_trees_equal(_trees(gpu), _trees(ref_ctx))
        got = _frames(gpu, built, sf, rects, n)
        _assert_frames_equal(got, _frames(ref_ctx, built, sf, rects, n))
        if edit == "deform":
            t = uo.with_trees(built, flat, p)
            o_rgb, o_hits, o_st = ob.render(t.ptr, sf.camera(), built.make_options(rects=rects, n_rects=n))
            rgb, hits, st = got[0]
            cov = _covered(sf, rects, n)
            assert same_f32(rgb, o_rgb).all(), edit
            assert np.array_equal(hits["mesh"][cov], o_hits["mesh"][cov]) and np.array_equal(hits["triangle"][cov], o_hits["triangle"][cov])
            assert [st[k] for k in RAY_KEYS] == [o_st[k] for k in RAY_KEYS]


def test_empty_scene(gpu, loaded, built, torch):
    """10 (n_vertices = 0): an empty scene updates to itself, with NULL positions."""
    sf, flat, rects, n = loaded["empty_scene"]
    assert flat.contents.n_vertices == 0
    gpu.upload(flat, keepalive=sf)
    before = _state(gpu)
    assert built.core().crtb200_update_vertices_device(gpu._h, None, 0, None) == 0
    _assert_state_equal(_state(gpu), before)
    gpu.update_vertices(torch.zeros((0, 3), dtype=torch.float32, device="cuda"))
    _assert_state_equal(_state(gpu), before)


def _overflowing(vp, verts):
    """Two vertices of one mesh at +-3.4e38: the root's extent overflows, a split plane is +inf and the mesh tree no
    longer nests."""
    p = vp.copy()
    p[verts[0]] = [3.4e38, 3.4e38, 3.4e38]
    p[verts[1]] = [-3.4e38, -3.4e38, -3.4e38]
    return p


def test_nesting_flips(gpu, ref_ctx, loaded, built, torch):
    """5: an edit that makes a mesh tree fail to nest (nested_ok 0, every margin +inf) and one that restores it."""
    sf, flat, rects, n = loaded["hw11_room"]
    vp = built.scene_vertex_positions(flat)
    gpu.upload(flat, keepalive=sf)
    assert gpu.debug_scene_layout()["nested_ok"]
    verts = _mesh_vertices(flat)[_largest_meshes(flat)[0]]
    for p, nested in ((_overflowing(vp, verts), False), (_deform(vp, 0.02), True)):
        _update(gpu, torch, p)
        e = uo.EditedScene(built, flat, p)
        ref_ctx.upload_geometry(e.ptr, keepalive=e)
        got = _state(gpu)
        _assert_state_equal(got, _state(ref_ctx))
        kb.assert_trees_equal(_trees(gpu), _trees(ref_ctx))
        assert got[0]["nested_ok"] == nested
        if not nested:
            assert np.isinf(got[0]["meshes"][:, 4].view(np.float32)).all()
        _assert_frames_equal(_frames(gpu, built, sf, rects, n), _frames(ref_ctx, built, sf, rects, n))


def test_animation_sequence(built, ref_ctx, loaded, torch):
    """6: ten successive deformations on one context, each equal to a fresh upload; device memory afterwards within the
    bound test_gpu_lifecycle.py allows."""
    from test_gpu_lifecycle import MAX_LOSS
    sf, flat, rects, n = loaded["hw14_small"]
    vp = built.scene_vertex_positions(flat)
    torch.cuda.synchronize()
    ctx = built.Context(0)
    try:
        ctx.upload_geometry(sf.flatten(trees=False), keepalive=sf)
        opt = built.make_options(rects=rects, n_rects=n)
        ctx.render(sf.camera(), opt)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        base = torch.from_numpy(vp).cuda()
        for f in range(10):
            ph = 0.6 * f
            d = base * (1.0 + 0.04 * torch.sin(3.0 * base[:, :1] + 2.0 * base[:, 1:2] + ph))
            ctx.update_vertices(d.contiguous())
            p = d.cpu().numpy()
            e = uo.EditedScene(built, flat, p)
            ref_ctx.upload_geometry(e.ptr, keepalive=e)
            _assert_state_equal(_state(ctx), _state(ref_ctx))
            a = ctx.render(sf.camera(), opt, want_hits=True)
            b = ref_ctx.render(sf.camera(), opt, want_hits=True)
            assert same_f32(a[0], b[0]).all() and np.array_equal(a[2]["triangle"], b[2]["triangle"]), f"frame {f}"
        torch.cuda.synchronize()
        free1 = torch.cuda.mem_get_info(0)[0]
        assert free0 - free1 < MAX_LOSS, f"ten updates lost {(free0 - free1) >> 20} MiB"
    finally:
        ctx.close()


def test_ordering_on_a_side_stream(gpu, loaded, built, torch):
    """7: positions written by a torch kernel on a non-default stream, then update_vertices on that stream at once: the
    written positions are the ones used."""
    sf, flat, _, _ = loaded["hw14_small"]
    vp = built.scene_vertex_positions(flat)
    gpu.upload(flat, keepalive=sf)
    new = _deform(vp, 0.08, 1.0)
    src = torch.from_numpy(new).cuda()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        dst = torch.zeros_like(src)
        torch.cuda._sleep(200_000_000)  # the write below lands well after the call is made
        dst.copy_(src)
        gpu.update_vertices(dst)
    fn, vn = uo.mesh_normals(new, kb.scene_arrays(flat)["triangle_vertex"])
    geom, got_vn = gpu.debug_scene_geometry()
    assert same_f32(geom, uo.tri_geom(new, kb.scene_arrays(flat)["triangle_vertex"], fn)).all()
    assert same_f32(got_vn, vn).all()


def test_side_effects(gpu, loaded, built, ob, torch):
    """8: a progressive session ends; pixels outside a later render's rects keep the colour buffer; last_stats and
    query_stats are unchanged; trace and shade answer for the new geometry (CPU oracle)."""
    core = built.core()
    sf, flat, rects, n = loaded["hw11_room"]
    vp = built.scene_vertex_positions(flat)
    gpu.upload(flat, keepalive=sf)
    p = gpu.progressive(sf.camera(), built.make_options(rects=rects, n_rects=n), built.Sampling.make())
    p.step(1)
    full, _, _, _ = gpu.render(sf.camera(), built.make_options())
    rays, md = caller_rays(flat, 1024, seed=3)
    d_rays = torch.from_numpy(rays).cuda()
    gpu.trace(d_rays, built.RAY_PRIMARY)
    q_before = gpu.query_stats()
    st_before = gpu.last_stats()
    new = _deform(vp, 0.05, 0.5)
    _update(gpu, torch, new)
    assert core.crtb200_accum_step(gpu._h, 1, None) == ERR_STATE
    assert gpu.last_stats() == st_before and gpu.query_stats() == q_before
    rect = (built.Rect * 1)()
    rect[0].row, rect[0].col, rect[0].width, rect[0].height = 8, 16, 40, 24
    part, _, _, _ = gpu.render(sf.camera(), built.make_options(rects=rect, n_rects=1))
    outside = np.ones(part.shape[:2], bool)
    outside[8:32, 16:56] = False
    assert same_f32(part[outside], full[outside]).all()
    t = uo.with_trees(built, flat, new)
    o_rgb, _, _ = ob.render(t.ptr, sf.camera(), built.make_options(rects=rect, n_rects=1))
    assert same_f32(part[~outside], o_rgb[~outside]).all()
    h = gpu.trace(d_rays, built.RAY_PRIMARY)
    oh = ob.trace_rays(t.ptr, rays, built.RAY_PRIMARY)
    got = np.ascontiguousarray(h.records.cpu().numpy()).view(ob.HIT_DTYPE)[..., 0]
    assert np.array_equal(got["mesh"], oh["mesh"]) and np.array_equal(got["triangle"], oh["triangle"])
    assert same_f32(got["t"], oh["t"]).all()
    occ = gpu.trace(d_rays, built.RAY_SHADOW, max_distance=torch.from_numpy(md).cuda())
    assert np.array_equal(occ.cpu().numpy(), ob.trace_rays(t.ptr, rays, built.RAY_SHADOW, md))
    rgb, _ = gpu.shade(d_rays, built.RAY_PRIMARY)
    o_rgb, _, _ = so.shade_rays(t.ptr, rays, built.RAY_PRIMARY, built.make_options())
    assert same_f32(rgb.cpu().numpy(), o_rgb).all()


def test_several_gpus(gpu, loaded, built, torch):
    """9: on Context([0, 0, 0]) every replica equals the single-GPU context after the same update, and frames are equal."""
    sf, flat, rects, n = loaded["hw14_small"]
    new = _deform(built.scene_vertex_positions(flat), 0.06, 2.0)
    gpu.upload(flat, keepalive=sf)
    _update(gpu, torch, new)
    one = _state(gpu)
    one_trees = _trees(gpu)
    one_frames = _frames(gpu, built, sf, rects, n)
    multi = built.Context([0, 0, 0])
    try:
        multi.upload_geometry(sf.flatten(trees=False), keepalive=sf)
        _update(multi, torch, new)
        for d in range(3):
            _assert_state_equal(_state(multi, d), one)
        kb.assert_trees_equal(_trees(multi), one_trees)
        _assert_frames_equal(_frames(multi, built, sf, rects, n), one_frames, ignore=("kernel_launches",))
    finally:
        multi.close()


def test_errors(built, loaded, torch):
    """10: no scene, null / host / misaligned positions, a wrong n_vertices, and the Python checks."""
    core = built.core()
    ctx = built.Context(0)
    try:
        buf = torch.zeros(3 * 1024 + 1, dtype=torch.float32, device="cuda")
        assert core.crtb200_update_vertices_device(ctx._h, buf.data_ptr(), 0, None) == ERR_STATE  # no scene
        sf, flat, _, _ = loaded["hw07_scene0"]
        ctx.upload(flat, keepalive=sf)
        V = flat.contents.n_vertices
        pos = torch.from_numpy(built.scene_vertex_positions(flat)).cuda()
        assert core.crtb200_update_vertices_device(ctx._h, None, V, None) == ERR_ARG
        host = built.scene_vertex_positions(flat)
        assert core.crtb200_update_vertices_device(ctx._h, host.ctypes.data, V, None) == ERR_ARG
        big = torch.zeros(3 * V + 1, dtype=torch.float32, device="cuda")
        assert core.crtb200_update_vertices_device(ctx._h, big.data_ptr() + 2, V, None) == ERR_ARG
        assert core.crtb200_update_vertices_device(ctx._h, pos.data_ptr(), V + 1, None) == ERR_ARG
        assert core.crtb200_update_vertices_device(ctx._h, pos.data_ptr(), V - 1, None) == ERR_ARG
        assert core.crtb200_update_vertices_device(None, pos.data_ptr(), V, None) == ERR_ARG
        # the checks leave the scene in place
        before = _state(ctx)
        assert core.crtb200_update_vertices_device(ctx._h, pos.data_ptr(), V, None) == 0
        _assert_state_equal(_state(ctx), before)
        for bad in (pos.double(), pos.cpu(), pos[:-1], pos.t().contiguous().t(), pos.reshape(-1)):
            with pytest.raises(built.CrtError):
                ctx.update_vertices(bad)
        t = built.Trees()
        assert core.crtb200_scene_trees(ctx._h, C.byref(t)) == 0  # an update's trees are device-built
    finally:
        ctx.close()


def test_full_size(gpu, ref_ctx, built, bench_mod, torch):
    """11: hw14_dragon_class with its sphere displaced by a torch kernel: the update's state equals upload_geometry of the
    edited host arrays."""
    sf, f, folder, tex, depth = _load(bench_mod, built, "hw14_dragon_class")
    geo = sf.flatten(trees=False)
    gpu.upload_geometry(geo, keepalive=sf)
    base = torch.from_numpy(built.scene_vertex_positions(geo)).cuda()
    d = base * (1.0 + 0.03 * torch.sin(5.0 * base[:, :1] + 3.0 * base[:, 2:3]))
    gpu.update_vertices(d.contiguous())
    e = uo.EditedScene(built, geo, d.cpu().numpy())
    ref_ctx.upload_geometry(e.ptr, keepalive=e)
    _assert_state_equal(_state(gpu), _state(ref_ctx))
    kb.assert_trees_equal(_trees(gpu), _trees(ref_ctx))


@pytest.fixture(scope="module")
def bench_mod():
    import importlib
    return importlib.import_module("bench")
