"""GI and jittered supersampling on the GPU (sampling contract, DESIGN.md 3.10): bit-identical to the CPU restatement
(tests/gi_oracle.c), independent of chunking, concurrency, tile shards and GPU count, and no change at all with sampling
off."""
import importlib
import os

import numpy as np
import pytest

import gi_oracle as gio
from conftest import SMALL_SCENES, same_f32
from handoff_contexts import HANDOFF, HandoffContexts
from test_sampling_oracle import unit_scenes  # noqa: F401 (fixture)

pytestmark = pytest.mark.gpu
CONFIGS = [dict(spp=2, G=1, depth=5), dict(spp=1, G=2, depth=3)]
RAYS = ("rays_primary", "rays_shadow", "rays_reflection", "rays_refraction")


@pytest.fixture(scope="module")
def gpu(built):
    try:
        ctx = built.Context(0)
    except built.CrtError as e:
        pytest.fail(f"CUDA core unusable on a GPU box: {e}")
    yield ctx
    ctx.close()


def _smp(crt, cfg, seed=11, frame_index=0):
    return crt.Sampling.make(gi_samples=cfg["G"], rays_per_pixel=cfg["spp"], seed=seed, frame_index=frame_index)


def _render(ctx, crt, sf, flat, cfg, seed=11, **opt_kw):
    ctx.upload(flat, keepalive=sf)
    ctx.set_sampling(_smp(crt, cfg, seed))
    rgb, rgb8, hits, st = ctx.render(sf.camera(), crt.make_options(max_depth=cfg["depth"], **opt_kw), want_rgb8=True, want_hits=True)
    st.update(ctx.sampling_stats())
    ctx.set_sampling(None)
    return rgb, rgb8, hits, st


@pytest.fixture(scope="module")
def handoff(built):
    """Contexts with the tail hand-off forced or off (handoff_contexts.HANDOFF_ENV), created on first use."""
    hc = HandoffContexts(built)
    yield hc
    hc.close()


_ORACLE = {}  # (scene, config) -> the CPU restatement's frame, shared by the hand-off contexts


def _oracle(name, ci, loaded, crt):
    if (name, ci) not in _ORACLE:
        sf, flat, rects, n = loaded[name]
        cfg = CONFIGS[ci]
        opt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n)
        _ORACLE[name, ci] = gio.render_sampled(flat, sf.camera(), opt, _smp(crt, cfg))
    return _ORACLE[name, ci]


@pytest.mark.parametrize("which", HANDOFF)
@pytest.mark.parametrize("ci", [0, 1], ids=["spp2_G1_d5", "spp1_G2_d3"])
@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_gi_matches_oracle(name, ci, which, handoff, loaded, ob, crt):
    """GI frames in every hand-off context (handoff_contexts.HANDOFF_ENV) against the CPU restatement: handed-off primary
    walks rebuild their jittered ray in k_coop, and handed-off shadow walks of a GI frame stop at refractive meshes."""
    sf, flat, rects, n = loaded[name]
    cfg = CONFIGS[ci]
    o_rgb, o_hits, o_st = _oracle(name, ci, loaded, crt)
    ctx = handoff(which)  # upload() clears the colour buffer: uncovered pixels stay 0 like the oracle's
    cov = np.zeros(o_hits.shape, bool)
    for i in range(n):
        r = rects[i]
        cov[r.row:r.row + r.height, r.col:r.col + r.width] = True
    for traversal in (0, 1):
        rgb, rgb8, hits, st = _render(ctx, crt, sf, flat, cfg, rects=rects, n_rects=n, traversal=traversal)
        same = same_f32(rgb, o_rgb)
        assert same.all(), f"{name} traversal {traversal}: {(~same).sum()} components differ"
        assert np.array_equal(rgb8, ob.quantize(rgb))
        assert np.array_equal(hits["mesh"][cov], o_hits["mesh"][cov]) and np.array_equal(hits["triangle"][cov], o_hits["triangle"][cov])
        for k in RAYS + ("rays_diffuse",):
            assert st[k] == o_st[k], (name, traversal, k, st[k], o_st[k])
        assert st["samples"] == cfg["spp"]
        if traversal == 0:
            if which in ("all", "final_only", "capped") and name != "empty_scene":
                assert st["handoff_closest"] > 0
                if o_st["rays_shadow"] > st["shadow_rays_zero_term"]:
                    assert st["handoff_shadow"] > 0
            if which == "off":
                assert st["handoff_closest"] == 0 and st["handoff_shadow"] == 0
    _, _, _, st = _render(ctx, crt, sf, flat, cfg, rects=rects, n_rects=n, count_work=1)
    for k in ("node_tests_closest", "triangle_tests_closest", "node_tests_shadow", "triangle_tests_shadow"):
        assert st[k] == o_st[k], (name, k, st[k], o_st[k])


def test_refractive_occluders_in_handed_off_gi_shadow_walks(handoff, unit_scenes, ob, crt):
    """The glass slab between the light and a diffuse floor, every walk handed off to k_coop, seen from below the slab
    looking straight down: every pixel is floor whose shadow ray crosses the slab, so every handed-off shadow walk is one
    the slab decides.  GI frames: refractive meshes cast shadows, the image is black; without sampling they do not
    (RayTracer.cpp's shadow rays skip them), every pixel is lit.  Pins the refractive-mesh rule of both k_coop shadow
    instantiations."""
    sf, flat = unit_scenes["glass"]
    cam = crt.Camera.make((0.0, -1.0, -5.0), (1, 0, 0, 0, 0, -1, 0, 1, 0))  # 0.8 above the floor, inside the slab's shadow
    ctx = handoff("all")
    ctx.upload(flat, keepalive=sf)
    opt = crt.make_options(max_depth=2)
    smp = crt.Sampling.make(gi_samples=0)
    ctx.set_sampling(smp)
    on, _, _, st = ctx.render(cam, opt)
    ctx.set_sampling(None)
    o_on, _, _ = gio.render_sampled(flat, cam, opt, smp, want_hits=False)
    assert st["handoff_shadow"] > 0
    assert (o_on == 0).all() and same_f32(on, o_on).all(), f"{(on != 0).any(axis=2).sum()} pixels lit through the slab"
    off, _, _, st = ctx.render(cam, opt)
    o_off, _, _ = ob.render(flat, cam, opt, want_hits=False)
    assert st["handoff_shadow"] > 0
    assert (o_off > 0).all() and same_f32(off, o_off).all(), f"{(off == 0).any(axis=2).sum()} pixels shadowed by the slab"


def test_gi_invariance(gpu, loaded, crt):
    torch = pytest.importorskip("torch")
    sf, flat, _, _ = loaded["hw11_room"]
    cfg = CONFIGS[0]
    ref, _, _, st = _render(gpu, crt, sf, flat, cfg)
    assert st["rays_diffuse"] > 0
    for conc in (1, 2):
        gpu.set_concurrency(conc)
        assert same_f32(_render(gpu, crt, sf, flat, cfg)[0], ref).all(), conc
    gpu.set_queue_budget(64 << 20)  # >= 3 chunks at this depth
    assert same_f32(_render(gpu, crt, sf, flat, cfg)[0], ref).all()
    gpu.set_queue_budget(16 << 30)
    # tile shards: compact slabs + assemble
    gpu.upload(flat, keepalive=sf)
    gpu.set_sampling(_smp(crt, cfg))
    world, items = 3, gpu.shard_items(3)
    slabs = torch.zeros((world, items, 3), dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    for r in range(world):
        gpu.render_device(sf.camera(), crt.make_options(max_depth=cfg["depth"], shard_index=r, shard_count=world),
                          d_rgb=slabs[r].data_ptr(), stream=stream)
    out = torch.zeros((sf.info.height, sf.info.width, 3), dtype=torch.float32, device="cuda")
    gpu.assemble_shards(slabs.data_ptr(), world, d_rgb=out.data_ptr(), stream=stream)
    torch.cuda.synchronize()
    assert same_f32(out.cpu().numpy(), ref).all()
    # render_frames: frame f is keyed frame_index + f
    cams = [sf.camera()] * 3
    frames, _, _ = gpu.render_frames(cams, crt.make_options(max_depth=cfg["depth"]))
    gpu.set_sampling(None)
    for f in range(3):
        gpu.set_sampling(_smp(crt, cfg, frame_index=f))
        one, _, _, _ = gpu.render(sf.camera(), crt.make_options(max_depth=cfg["depth"]))
        assert same_f32(frames[f], one).all(), f
    gpu.set_sampling(None)
    assert not same_f32(frames[0], frames[1]).all()
    assert not same_f32(_render(gpu, crt, sf, flat, cfg, seed=12)[0], ref).all()
    multi = crt.Context([0, 0, 0])
    try:
        assert same_f32(_render(multi, crt, sf, flat, cfg)[0], ref).all()
        # settings changed after creation hold on every GPU of the context
        multi.set_concurrency(1)
        multi.set_queue_budget(64 << 20)
        assert same_f32(_render(multi, crt, sf, flat, cfg)[0], ref).all()
        multi.set_queue_budget(16 << 30)
        multi.set_concurrency(2)
        # pipelined render_frames: every GPU keys frame f with frame_index + f
        multi.set_sampling(_smp(crt, cfg))
        mframes, _, _ = multi.render_frames(cams, crt.make_options(max_depth=cfg["depth"]))
        multi.set_sampling(None)
        for f in range(3):
            assert same_f32(mframes[f], frames[f]).all(), f
    finally:
        multi.close()


def test_sampling_off_is_unchanged(gpu, loaded, crt):
    sf, flat, rects, n = loaded["hw11_room"]
    opt = crt.make_options(rects=rects, n_rects=n)
    fresh = crt.Context(0)
    try:
        fresh.upload(flat, keepalive=sf)
        a, a8, ha, sa = fresh.render(sf.camera(), opt, want_rgb8=True, want_hits=True)
    finally:
        fresh.close()
    _render(gpu, crt, sf, flat, CONFIGS[1])  # sampling on, then off
    b, b8, hb, sb = gpu.render(sf.camera(), opt, want_rgb8=True, want_hits=True)
    assert a.tobytes() == b.tobytes() and np.array_equal(a8, b8) and ha.tobytes() == hb.tobytes()
    assert all(sa[k] == sb[k] for k in RAYS) and gpu.sampling_stats() == {"rays_diffuse": 0, "samples": 1}


def test_front_end_and_errors(gpu, loaded, crt):
    sf, flat, _, _ = loaded["hw11_room"]
    tracer = crt.RayTracer(sf, device=0)
    try:
        rgb, st = tracer.render(max_depth=3, use_gi=True, gi_samples=2, rays_per_pixel=2, seed=4)
    finally:
        tracer.close()
    rects, n = sf.rects(mode=crt.MODE_B200_WAVEFRONT)
    ctx = crt.Context(0)
    try:
        ctx.upload(flat, keepalive=sf)
        ctx.set_sampling(crt.Sampling.make(gi_samples=2, rays_per_pixel=2, seed=4))
        want, _, _, _ = ctx.render(sf.camera(), crt.make_options(max_depth=3, rects=rects, n_rects=n))
        assert same_f32(rgb, want).all()
        ctx.set_sampling(crt.Sampling.make(gi_samples=64, rays_per_pixel=1))
        with pytest.raises(crt.CrtError, match="error -4"):
            ctx.render(sf.camera(), crt.make_options(max_depth=5))
        with pytest.raises(crt.CrtError, match="error -1"):
            ctx.set_sampling(crt.Sampling.make(rays_per_pixel=0))
        with pytest.raises(crt.CrtError, match="error -1"):
            ctx.set_sampling(crt.Sampling.make(gi_samples=1025))
    finally:
        ctx.close()


def test_full_size_room(gpu, built, scenes_mod, tmp_path):
    d = str(tmp_path)
    scenes_mod.write_crtscene(os.path.join(d, "room.crtscene"), scenes_mod.hw11_room())
    sf = built.SceneFile("room.crtscene", d)
    flat = sf.flatten()
    cfg = dict(spp=8, G=1, depth=5)
    rgb, _, _, _ = _render(gpu, built, sf, flat, cfg)
    gpu.set_queue_budget(256 << 20)
    chunked, _, _, _ = _render(gpu, built, sf, flat, cfg)
    gpu.set_queue_budget(16 << 30)
    assert same_f32(rgb, chunked).all()
    rects, n = sf.rects()
    picked = (built.Rect * 2)(rects[7], rects[16])  # two of the 24 buckets; keys are global, so a crop is exact
    o_rgb, _, _ = gio.render_sampled(flat, sf.camera(), built.make_options(max_depth=5, rects=picked, n_rects=2), _smp(built, cfg),
                                     want_hits=False)
    for r in picked:
        win = (slice(r.row, r.row + r.height), slice(r.col, r.col + r.width))
        assert same_f32(rgb[win], o_rgb[win]).all(), (r.row, r.col)


def test_4k_dragon_gi(handoff, built, crt):
    """hw14_dragon_class at its stated size (3840x2160, 1 009 202 triangles: the long walks) as a GI frame.  The host path
    (several chunk streams, dynamic thresholds) against the CPU restatement on two windows -- one inside the dragon, one
    across its silhouette (keys are global, so a crop is exact) -- and the whole frame bit-identical through one stream
    (render_device: k_coop's early pass runs), the literal walk, and the "mid" and "capped" hand-off contexts."""
    torch = pytest.importorskip("torch")
    f, folder, _, _, _ = importlib.import_module("bench").ensure_scene("hw14_dragon_class", {})
    sf = built.SceneFile(f, folder)
    flat = sf.flatten()
    W, H = sf.info.width, sf.info.height
    assert (W, H) == (3840, 2160)
    cfg = dict(spp=2, G=1, depth=5)
    ctx = handoff("default")
    rgb, _, hits, st = _render(ctx, crt, sf, flat, cfg)
    assert st["rays_diffuse"] > 0
    s = flat.contents
    dragon = max(range(s.n_meshes), key=lambda m: s.meshes[m].n_nodes)
    ys, xs = np.nonzero(hits["mesh"] == dragon)
    top = int(ys.min())
    # 64x32 windows on the 8x4 tile grid: around the dragon's centroid, and around the top of its outline (sky above)
    wins = [((int(ys.mean()) - 16) // 4 * 4, (int(xs.mean()) - 32) // 8 * 8),
            ((top - 16) // 4 * 4, (int(xs[ys == top].mean()) - 32) // 8 * 8)]
    picked = (crt.Rect * 2)(*[crt.Rect(row=r, col=c, width=64, height=32) for r, c in wins])
    o_rgb, o_hits, _ = gio.render_sampled(flat, sf.camera(), crt.make_options(max_depth=cfg["depth"], rects=picked, n_rects=2),
                                          _smp(crt, cfg))
    for k, (r, c) in enumerate(wins):
        win = (slice(r, r + 32), slice(c, c + 64))
        mesh = o_hits["mesh"][win]
        assert (mesh == dragon).all() if k == 0 else ((mesh == dragon).any() and (mesh < 0).any()), (r, c)
        assert np.array_equal(hits["mesh"][win], mesh) and np.array_equal(hits["triangle"][win], o_hits["triangle"][win]), (r, c)
        same = same_f32(rgb[win], o_rgb[win])
        assert same.all(), f"window ({r}, {c}): {(~same).sum()} components differ"
    # whole-frame variants
    out = torch.zeros((H, W, 3), dtype=torch.float32, device="cuda")
    ctx.set_sampling(_smp(crt, cfg))
    ctx.render_device(sf.camera(), crt.make_options(max_depth=cfg["depth"]), d_rgb=out.data_ptr(),
                      stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ctx.set_sampling(None)
    variants = [("render_device", out.cpu().numpy(), None),
                ("traversal 1",) + tuple(_render(ctx, crt, sf, flat, cfg, traversal=1)[::3])]
    for which in ("mid", "capped"):
        variants.append((which,) + tuple(_render(handoff(which), crt, sf, flat, cfg)[::3]))
    for what, got, vst in variants:
        same = same_f32(got, rgb)
        assert same.all(), f"{what}: {(~same).sum()} components differ"
        if vst is not None:
            assert all(vst[k] == st[k] for k in RAYS + ("rays_diffuse",)), what
            if what != "traversal 1":
                assert vst["handoff_closest"] > 0 and vst["handoff_shadow"] > 0, what
