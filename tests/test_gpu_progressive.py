"""Progressive GI sessions on the GPU (DESIGN.md 3.10.1): after steps totalling n samples the read is bit-identical to
the one-shot frame with rays_per_pixel = n, ray and test counts add up, the accumulator equals the CPU restatement's,
and sessions survive save / resume, chunking, concurrency, GPU lists and renders in between."""
import os

import numpy as np
import pytest

import progressive_oracle as po
from conftest import SMALL_SCENES, same_f32
from handoff_contexts import handoff_context

pytestmark = pytest.mark.gpu
CONFIGS = [dict(G=1, depth=5), dict(G=2, depth=3)]
RAYS = ("rays_primary", "rays_shadow", "rays_reflection", "rays_refraction", "rays_diffuse")
TESTS = ("node_tests_closest", "triangle_tests_closest", "node_tests_shadow", "triangle_tests_shadow")


def _smp(crt, cfg, spp=1, seed=11):
    return crt.Sampling.make(gi_samples=cfg["G"], rays_per_pixel=spp, seed=seed)


def _oneshot(ctx, crt, sf, cfg, spp, opt, seed=11):
    ctx.set_sampling(_smp(crt, cfg, spp, seed))
    rgb, rgb8, hits, st = ctx.render(sf.camera(), opt, want_rgb8=True, want_hits=True)
    st.update(ctx.sampling_stats())
    ctx.set_sampling(None)
    return rgb, rgb8, hits, st


def _covered(shape, rects, n):
    cov = np.zeros(shape, bool) if n else np.ones(shape, bool)
    for i in range(n):
        r = rects[i]
        cov[r.row:r.row + r.height, r.col:r.col + r.width] = True
    return cov


def _same_frame(got, want, cov):
    rgb, rgb8, hits = got
    w_rgb, w_rgb8, w_hits = want[:3]
    assert same_f32(rgb, w_rgb).all(), f"{(~same_f32(rgb, w_rgb)).sum()} components differ"
    assert np.array_equal(rgb8, w_rgb8)
    assert np.array_equal(hits["mesh"][cov], w_hits["mesh"][cov]) and np.array_equal(hits["triangle"][cov], w_hits["triangle"][cov])
    hit = cov & (w_hits["mesh"] >= 0)
    assert same_f32(hits["t"][hit], w_hits["t"][hit]).all()


def _context(crt, sf, flat, devices=0, handoff="default"):
    """A context holding the scene; `handoff` names the tail hand-off setting (handoff_contexts.HANDOFF_ENV)."""
    ctx = handoff_context(crt, handoff, devices)
    ctx.upload(flat, keepalive=sf)
    return ctx


@pytest.mark.parametrize("cfg", CONFIGS, ids=["G1_d5", "G2_d3"])
@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_prefix_exactness(name, cfg, loaded, crt):
    sf, flat, rects, n = loaded[name]
    opt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n)
    cnt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n, count_work=1)
    one, ses = _context(crt, sf, flat), _context(crt, sf, flat)
    try:
        p = ses.progressive(sf.camera(), opt, _smp(crt, cfg, spp=5))  # rays_per_pixel is ignored
        total = dict.fromkeys(RAYS, 0)
        for step, spp in ((1, 1), (3, 4), (4, 8)):
            st = p.step(step)
            assert p.samples == spp and st["samples"] == step
            for k in RAYS:
                total[k] += st[k]
            want = _oneshot(one, crt, sf, cfg, spp, opt)
            _same_frame(p.read(want_rgb8=True, want_hits=True), want, _covered((sf.info.height, sf.info.width), rects, n))
            for k in RAYS:
                assert total[k] == want[3][k], (name, spp, k, total[k], want[3][k])
        p.close()
        p = ses.progressive(sf.camera(), cnt, _smp(crt, cfg))
        total = dict.fromkeys(RAYS + TESTS, 0)
        for step in (1, 3, 4):
            st = p.step(step)
            for k in total:
                total[k] += st[k]
        want = _oneshot(one, crt, sf, cfg, 8, cnt)
        for k in total:
            assert total[k] == want[3][k], (name, "count_work", k, total[k], want[3][k])
        assert same_f32(p.read()[0], want[0]).all()
    finally:
        one.close()
        ses.close()


@pytest.mark.parametrize("name", ["hw11_room", "hw12_textures", "degenerate_uv"])
def test_sums_match_oracle(name, loaded, crt):
    sf, flat, rects, n = loaded[name]
    cfg = CONFIGS[0]
    opt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n)
    o_sum, o_sumsq = po.render_sums(flat, sf.camera(), opt, _smp(crt, cfg, spp=4))
    ctx = _context(crt, sf, flat)
    try:
        p = ctx.progressive(sf.camera(), opt, _smp(crt, cfg))
        p.step(1)
        p.step(3)
        a = p.arrays()
        assert int(a["samples"]) == 4
        assert same_f32(a["sum"], o_sum).all() and same_f32(a["sumsq"], o_sumsq).all()
        se = p.std_error()
        assert se.shape == o_sum.shape and not (se < 0).any()
    finally:
        ctx.close()


def _session_bits(ctx, crt, sf, opt, cfg):
    p = ctx.progressive(sf.camera(), opt, _smp(crt, cfg))
    p.step(3)
    p.step(5)
    rgb = p.read()[0]
    a = p.arrays()
    p.close()
    return rgb, a


def test_invariance(loaded, crt):
    sf, flat, _, _ = loaded["hw11_room"]
    cfg = CONFIGS[0]
    opt = crt.make_options(max_depth=cfg["depth"])
    ctx = _context(crt, sf, flat)
    try:
        ref, ref_a = _session_bits(ctx, crt, sf, opt, cfg)
        variants = []
        for conc in (1, 2):
            ctx.set_concurrency(conc)
            variants.append((f"concurrency {conc}", _session_bits(ctx, crt, sf, opt, cfg)))
        ctx.set_queue_budget(64 << 20)  # several chunks at this depth
        variants.append(("64 MiB queues", _session_bits(ctx, crt, sf, opt, cfg)))
        ctx.set_queue_budget(16 << 30)
        variants.append(("traversal 1", _session_bits(ctx, crt, sf, crt.make_options(max_depth=cfg["depth"], traversal=1), cfg)))
    finally:
        ctx.close()
    for which, devices in (("default", [0, 0, 0]), ("all", 0), ("mid", 0), ("capped", 0), ("mid", [0, 0, 0])):
        ctx = _context(crt, sf, flat, devices, which)
        try:
            variants.append((f"Context({devices}), hand-off {which}", _session_bits(ctx, crt, sf, opt, cfg)))
        finally:
            ctx.close()
    for what, (rgb, a) in variants:
        assert same_f32(rgb, ref).all(), what
        for k in ("sum", "sumsq"):
            assert same_f32(a[k], ref_a[k]).all(), (what, k)
        assert a["hit0"].tobytes() == ref_a["hit0"].tobytes(), what


@pytest.mark.parametrize("devices", [(0, 0), (0, [0, 0, 0]), ([0, 0, 0], 0)], ids=["single", "single_to_multi", "multi_to_single"])
def test_save_resume(devices, loaded, crt, tmp_path):
    sf, flat, rects, n = loaded["hw12_textures"]
    cfg = CONFIGS[0]
    opt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n)
    path = str(tmp_path / "session.npz")
    ctx = _context(crt, sf, flat, devices[0])
    try:
        p = ctx.progressive(sf.camera(), opt, _smp(crt, cfg))
        p.step(4)
        p.save(path)
        assert np.isnan(ctx.progressive(sf.camera(), opt, _smp(crt, cfg)).std_error()).all()  # 0 samples
    finally:
        ctx.close()
    ctx = _context(crt, sf, flat, devices[1])
    try:
        p = ctx.resume(path, sf.camera(), opt, _smp(crt, cfg, spp=3))
        assert p.samples == 4
        p.step(4)
        got = p.read(want_rgb8=True, want_hits=True)
        want = _oneshot(ctx, crt, sf, cfg, 8, opt)
        _same_frame(got, want, _covered((sf.info.height, sf.info.width), rects, n))
        moved = sf.camera()
        moved.position[0] += 0.5
        for cam, o, smp in ((sf.camera(), opt, _smp(crt, cfg, seed=12)), (moved, opt, _smp(crt, cfg)),
                            (sf.camera(), crt.make_options(max_depth=4, rects=rects, n_rects=n), _smp(crt, cfg))):
            with pytest.raises(crt.CrtError, match="differs"):
                ctx.resume(path, cam, o, smp)
    finally:
        ctx.close()


def test_isolation_and_errors(loaded, crt):
    sf, flat, rects, n = loaded["hw11_room"]
    cfg = CONFIGS[1]
    opt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n)
    ctx = _context(crt, sf, flat)
    try:
        lib = crt.core()
        with pytest.raises(crt.CrtError, match="error -3"):
            crt._check_core(lib.crtb200_accum_step(ctx._h, 1, None))
        with pytest.raises(crt.CrtError, match="error -3"):
            crt._check_core(lib.crtb200_accum_read(ctx._h, None, None, None, None))
        p = ctx.progressive(sf.camera(), opt, _smp(crt, cfg))
        with pytest.raises(crt.CrtError, match="error -3"):
            p.read()
        with pytest.raises(crt.CrtError, match="error -1"):
            p.step(0)
        p.step(2)
        ctx.set_sampling(crt.Sampling.make(gi_samples=1, rays_per_pixel=3, seed=99, frame_index=4))
        ctx.render(sf.camera(), crt.make_options(max_depth=2))
        ctx.set_sampling(crt.Sampling.make(gi_samples=3, rays_per_pixel=2, seed=7))
        p.step(2)
        got = p.read(want_rgb8=True, want_hits=True)
        want = _oneshot(ctx, crt, sf, cfg, 4, opt)
        _same_frame(got, want, _covered((sf.info.height, sf.info.width), rects, n))
        ctx.upload(flat, keepalive=sf)
        with pytest.raises(crt.CrtError, match="error -3"):
            p.step(1)
        with pytest.raises(crt.CrtError, match="error -1"):
            ctx.progressive(sf.camera(), opt, crt.Sampling.make(use_gi=False))
        with pytest.raises(crt.CrtError, match="error -1"):
            ctx.progressive(sf.camera(), crt.make_options(max_depth=3, shard_count=2), _smp(crt, cfg))
    finally:
        ctx.close()


def test_full_size_room(built, scenes_mod, tmp_path):
    d = str(tmp_path)
    scenes_mod.write_crtscene(os.path.join(d, "room.crtscene"), scenes_mod.hw11_room())
    sf = built.SceneFile("room.crtscene", d)
    flat = sf.flatten()
    cfg = dict(G=1, depth=5)
    opt = built.make_options(max_depth=5)
    ctx = _context(built, sf, flat)
    try:
        assert (sf.info.width, sf.info.height) == (1920, 1080)
        p = ctx.progressive(sf.camera(), opt, _smp(built, cfg))
        p.step(2)
        p.step(6)
        got = p.read(want_rgb8=True, want_hits=True)
        p.close()
        _same_frame(got, _oneshot(ctx, built, sf, cfg, 8, opt), np.ones((1080, 1920), bool))
    finally:
        ctx.close()
