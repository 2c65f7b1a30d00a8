"""GI and jittered supersampling on the GPU (sampling contract, DESIGN.md 3.10): bit-identical to the CPU restatement
(tests/gi_oracle.c), independent of chunking, concurrency, tile shards and GPU count, and no change at all with sampling
off."""
import os

import numpy as np
import pytest

import gi_oracle as gio
from conftest import SMALL_SCENES, same_f32

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


@pytest.mark.parametrize("cfg", CONFIGS, ids=["spp2_G1_d5", "spp1_G2_d3"])
@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_gi_matches_oracle(name, cfg, gpu, loaded, ob, crt):
    sf, flat, rects, n = loaded[name]
    smp = _smp(crt, cfg)
    opt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n)
    o_rgb, o_hits, o_st = gio.render_sampled(flat, sf.camera(), opt, smp)
    ctx = crt.Context(0)  # fresh colour buffer: uncovered pixels stay 0 like the oracle's
    try:
        for traversal in (0, 1):
            rgb, rgb8, hits, st = _render(ctx, crt, sf, flat, cfg, rects=rects, n_rects=n, traversal=traversal)
            same = same_f32(rgb, o_rgb)
            assert same.all(), f"{name} traversal {traversal}: {(~same).sum()} components differ"
            assert np.array_equal(rgb8, ob.quantize(rgb))
            for k in RAYS + ("rays_diffuse",):
                assert st[k] == o_st[k], (name, traversal, k, st[k], o_st[k])
            assert st["samples"] == cfg["spp"]
        cov = np.zeros(hits.shape, bool)
        for i in range(n):
            r = rects[i]
            cov[r.row:r.row + r.height, r.col:r.col + r.width] = True
        assert np.array_equal(hits["mesh"][cov], o_hits["mesh"][cov]) and np.array_equal(hits["triangle"][cov], o_hits["triangle"][cov])
        _, _, _, st = _render(ctx, crt, sf, flat, cfg, rects=rects, n_rects=n, count_work=1)
        for k in ("node_tests_closest", "triangle_tests_closest", "node_tests_shadow", "triangle_tests_shadow"):
            assert st[k] == o_st[k], (name, k, st[k], o_st[k])
    finally:
        ctx.close()


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
    multi = crt.Context([0, 0, 0])
    try:
        assert same_f32(_render(multi, crt, sf, flat, cfg)[0], ref).all()
    finally:
        multi.close()
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
