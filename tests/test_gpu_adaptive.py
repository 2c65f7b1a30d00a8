"""Adaptive progressive sessions on the GPU (DESIGN.md 3.10.2): each pixel stops once its noise is below the bound, and
pixel p of the session is bit for bit a plain session (and a one-shot frame) after n_p samples.  Counts, S, Q and ray
counts equal the CPU restatement's and do not depend on chunking, concurrency, queue budget, traversal or GPU list."""
import os

import numpy as np
import pytest

import adaptive_oracle as ao
from conftest import SMALL_SCENES, same_f32
from test_gpu_progressive import CONFIGS, RAYS, TESTS, _context, _covered, _oneshot, _smp

pytestmark = pytest.mark.gpu
PASSES = 14


def _ad(crt, mn=2, mx=12):
    return crt.Adaptive.make(min_samples=mn, max_samples=mx, abs_error=0.01, rel_error=0.03)


def _run(p, steps):
    total = dict.fromkeys(RAYS + TESTS, 0)
    for n in steps:
        st = p.step(n)
        for k in total:
            total[k] += st[k]
    return total


def _plain_at_counts(ctx, crt, sf, opt, cfg, counts):
    """A plain session's S / Q after n samples, at the pixels with counts == n, for every n in the map."""
    s = np.zeros(counts.shape + (3,), np.float32)
    q = np.zeros_like(s)
    p = ctx.progressive(sf.camera(), opt, _smp(crt, cfg))
    done = 0
    for n in np.unique(counts[counts > 0]):
        p.step(int(n) - done)
        done = int(n)
        a = p.arrays()
        m = counts == n
        s[m], q[m] = a["sum"][m], a["sumsq"][m]
    p.close()
    return s, q


@pytest.mark.parametrize("cfg", CONFIGS, ids=["G1_d5", "G2_d3"])
@pytest.mark.parametrize("name", list(SMALL_SCENES))
def test_prefix_exactness_and_oracle(name, cfg, loaded, crt):
    sf, flat, rects, n = loaded[name]
    opt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n)
    cnt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n, count_work=1)
    cov = _covered((sf.info.height, sf.info.width), rects, n)
    ctx, one = _context(crt, sf, flat), _context(crt, sf, flat)
    try:
        p = ctx.progressive(sf.camera(), opt, _smp(crt, cfg), _ad(crt))
        total = _run(p, (1, 3, 10))
        a = p.arrays()
        counts = a["counts"]
        got = p.read(want_rgb8=True, want_hits=True)
        pr = p.progress()
        p.close()
        assert (counts[~cov] == 0).all() and (counts[cov] >= 1).all() and counts.max() <= 12
        assert pr["passes"] == PASSES and pr["covered_pixels"] == cov.sum() and pr["pixel_samples"] == counts.sum()
        assert pr["active_pixels"] == 0  # max_samples 12 < 14 passes
        if name == "hw11_room":
            assert len(np.unique(counts[cov])) >= 3
        # per-pixel prefix exactness against a plain session
        ps, pq = _plain_at_counts(ctx, crt, sf, opt, cfg, counts)
        assert same_f32(a["sum"], ps).all() and same_f32(a["sumsq"], pq).all()
        # ... and against one-shot frames, for the smallest and largest counts present
        present = np.unique(counts[cov])
        for k in sorted({int(present.min()), int(present.max())}) if present.size else []:
            w_rgb, w_rgb8, w_hits, _ = _oneshot(one, crt, sf, cfg, k, opt)
            m = cov & (counts == k)
            assert same_f32(got[0][m], w_rgb[m]).all() and np.array_equal(got[1][m], w_rgb8[m]), (name, k)
            assert np.array_equal(got[2]["mesh"][m], w_hits["mesh"][m]) and np.array_equal(got[2]["triangle"][m], w_hits["triangle"][m])
            hit = m & (w_hits["mesh"] >= 0)
            assert same_f32(got[2]["t"][hit], w_hits["t"][hit]).all()
        # the CPU restatement: counts, S, Q and ray counts; with count_work = 1 the visit-all test counts
        o_s, o_q, o_c, o_st = ao.render_adaptive(flat, sf.camera(), opt, _smp(crt, cfg), _ad(crt), PASSES)
        assert np.array_equal(counts, o_c)
        assert same_f32(a["sum"], o_s).all() and same_f32(a["sumsq"], o_q).all()
        for k in RAYS:
            assert total[k] == o_st[k], (name, k, total[k], o_st[k])
        p = ctx.progressive(sf.camera(), cnt, _smp(crt, cfg), _ad(crt))
        total = _run(p, (5, 9))
        p.close()
        _, _, _, o_st = ao.render_adaptive(flat, sf.camera(), cnt, _smp(crt, cfg), _ad(crt), PASSES)
        for k in RAYS + TESTS:
            assert total[k] == o_st[k], (name, "count_work", k, total[k], o_st[k])
    finally:
        ctx.close()
        one.close()


def test_degenerate_equals_plain(loaded, crt):
    sf, flat, rects, n = loaded["hw12_textures"]
    cfg = CONFIGS[0]
    opt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n, count_work=1)
    ctx, two = _context(crt, sf, flat), _context(crt, sf, flat)
    try:
        a = ctx.progressive(sf.camera(), opt, _smp(crt, cfg), _ad(crt, 4, 4))
        p = two.progressive(sf.camera(), opt, _smp(crt, cfg))
        for step in (1, 2, 1):
            sa, sp = a.step(step), p.step(step)
            for k in RAYS + TESTS:
                assert sa[k] == sp[k], (step, k)
            assert sa["pixel_samples"] == sp["pixel_samples"]
            assert same_f32(a.read()[0], p.read()[0]).all()
            aa, pa = a.arrays(), p.arrays()
            for k in ("sum", "sumsq", "counts"):
                assert aa[k].tobytes() == pa[k].tobytes(), (step, k)
        assert a.progress()["active_pixels"] == 0
    finally:
        ctx.close()
        two.close()


def _bits(ctx, crt, sf, opt, cfg, steps):
    """The session's image and arrays, and the walks its steps handed off to k_coop (closest hit)."""
    p = ctx.progressive(sf.camera(), opt, _smp(crt, cfg), _ad(crt, 2, 8))
    handed_off = sum(p.step(s)["handoff_closest"] for s in steps)
    rgb = p.read()[0]
    a = p.arrays()
    p.close()
    return rgb, a, handed_off


def test_invariance(loaded, crt):
    sf, flat, _, _ = loaded["hw11_room"]
    cfg = CONFIGS[0]
    opt = crt.make_options(max_depth=cfg["depth"])
    ctx = _context(crt, sf, flat)
    try:
        ref = _bits(ctx, crt, sf, opt, cfg, (3, 5))
        variants = [("1 x 8", _bits(ctx, crt, sf, opt, cfg, (1,) * 8)), ("8", _bits(ctx, crt, sf, opt, cfg, (8,)))]
        for conc in (1, 2):
            ctx.set_concurrency(conc)
            variants.append((f"concurrency {conc}", _bits(ctx, crt, sf, opt, cfg, (3, 5))))
        ctx.set_queue_budget(64 << 20)
        variants.append(("64 MiB queues", _bits(ctx, crt, sf, opt, cfg, (3, 5))))
        ctx.set_queue_budget(16 << 30)
        variants.append(("traversal 1", _bits(ctx, crt, sf, crt.make_options(max_depth=cfg["depth"], traversal=1), cfg, (3, 5))))
    finally:
        ctx.close()
    # forced hand-off: k_coop maps the level-0 slots of handed-off primary walks through the pass's active list
    forced = []
    for which, devices in (("default", [0, 0, 0]), ("all", 0), ("mid", 0), ("capped", 0), ("mid", [0, 0, 0])):
        ctx = _context(crt, sf, flat, devices, which)
        try:
            variants.append((f"Context({devices}), hand-off {which}", _bits(ctx, crt, sf, opt, cfg, (3, 5))))
            if which != "default":
                forced.append(variants[-1])
        finally:
            ctx.close()
    assert len(np.unique(ref[1]["counts"])) >= 3
    for what, (rgb, a, _) in variants:
        assert same_f32(rgb, ref[0]).all(), what
        for k in ("sum", "sumsq", "counts"):
            assert same_f32(a[k].view(np.float32), ref[1][k].view(np.float32)).all(), (what, k)
    for what, (_, _, handed_off) in forced:
        assert handed_off > 0, what


@pytest.mark.parametrize("devices", [(0, 0), (0, [0, 0, 0]), ([0, 0, 0], 0)], ids=["single", "single_to_multi", "multi_to_single"])
def test_save_resume(devices, loaded, crt, tmp_path):
    sf, flat, rects, n = loaded["hw11_room"]
    cfg = CONFIGS[0]
    opt = crt.make_options(max_depth=cfg["depth"], rects=rects, n_rects=n)
    path, plain_path = str(tmp_path / "adaptive.npz"), str(tmp_path / "plain.npz")
    ctx = _context(crt, sf, flat, devices[0])
    try:
        p = ctx.progressive(sf.camera(), opt, _smp(crt, cfg), _ad(crt))
        p.step(5)
        mid = p.progress()
        assert 0 < mid["active_pixels"] < mid["covered_pixels"]  # mid-convergence
        p.save(path)
        q = ctx.progressive(sf.camera(), opt, _smp(crt, cfg))
        q.step(2)
        q.save(plain_path)
        ref = ctx.progressive(sf.camera(), opt, _smp(crt, cfg), _ad(crt))
        ref.step(PASSES)
        want, want_a = ref.read()[0], ref.arrays()
    finally:
        ctx.close()
    ctx = _context(crt, sf, flat, devices[1])
    try:
        p = ctx.resume(path, sf.camera(), opt, _smp(crt, cfg), _ad(crt))
        assert p.samples == 5 and p.progress() == mid
        p.step(PASSES - 5)
        a = p.arrays()
        assert same_f32(p.read()[0], want).all()
        for k in ("sum", "sumsq", "counts"):
            assert a[k].tobytes() == want_a[k].tobytes(), k
        with pytest.raises(crt.CrtError, match="plain"):
            ctx.resume(path, sf.camera(), opt, _smp(crt, cfg))
        with pytest.raises(crt.CrtError, match="adaptive"):
            ctx.resume(plain_path, sf.camera(), opt, _smp(crt, cfg), _ad(crt))
        with pytest.raises(crt.CrtError, match="adaptive parameters differ"):
            ctx.resume(path, sf.camera(), opt, _smp(crt, cfg), _ad(crt, 2, 13))
        with np.load(path) as f:
            data = {k: f[k] for k in f.files}
        for bad in (data["counts"] + np.uint32(1), data["counts"] * np.uint32(0), data["counts"][:-1]):
            broken = str(tmp_path / "broken.npz")
            np.savez(broken, **{**data, "counts": bad})
            with pytest.raises(crt.CrtError):
                ctx.resume(broken, sf.camera(), opt, _smp(crt, cfg), _ad(crt))
    finally:
        ctx.close()


def test_passes_after_convergence_trace_nothing(loaded, crt):
    sf, flat, rects, n = loaded["hw07_scene0"]
    ctx = _context(crt, sf, flat)
    try:
        p = ctx.progressive(sf.camera(), crt.make_options(max_depth=3, rects=rects, n_rects=n), _smp(crt, CONFIGS[1]),
                            _ad(crt, 2, 6))
        steps = p.run(passes_per_step=4)
        assert steps and steps[-1]["active_pixels"] == 0
        before = p.arrays()
        st = p.step(3)
        assert sum(st[k] for k in RAYS) == 0 and st["pixel_samples"] == before["counts"].sum()
        after = p.arrays()
        for k in ("sum", "sumsq", "counts"):
            assert after[k].tobytes() == before[k].tobytes(), k
    finally:
        ctx.close()


def test_rects_keep_the_context_buffer(loaded, crt):
    sf, flat, rects, n = loaded["uncovered"]
    assert n
    cov = _covered((sf.info.height, sf.info.width), rects, n)
    ctx = _context(crt, sf, flat)
    try:
        full, _, _, _ = ctx.render(sf.camera(), crt.make_options(max_depth=2))
        p = ctx.progressive(sf.camera(), crt.make_options(max_depth=3, rects=rects, n_rects=n), _smp(crt, CONFIGS[0]), _ad(crt))
        p.step(6)
        counts = p.counts()
        rgb = p.read()[0]
        assert (counts[~cov] == 0).all() and (counts[cov] > 0).all()
        assert same_f32(rgb[~cov], full[~cov]).all()
    finally:
        ctx.close()


def test_errors(loaded, crt):
    sf, flat, _, _ = loaded["hw11_room"]
    opt = crt.make_options(max_depth=3)
    ctx = _context(crt, sf, flat)
    try:
        with pytest.raises(crt.CrtError, match="error -3"):
            crt._check_core(crt.core().crtb200_accum_progress(ctx._h, crt.AccumProgress()))
        with pytest.raises(crt.CrtError, match="error -3"):
            crt._check_core(crt.core().crtb200_accum_counts(ctx._h, np.zeros(sf.info.width * sf.info.height, np.uint32).ctypes.data))
        bad = [crt.Adaptive.make(min_samples=1), crt.Adaptive.make(min_samples=8, max_samples=7),
               crt.Adaptive.make(abs_error=-0.1), crt.Adaptive.make(rel_error=float("nan"))]
        for ad in bad:
            with pytest.raises(crt.CrtError, match="error -1"):
                ctx.progressive(sf.camera(), opt, _smp(crt, CONFIGS[0]), ad)
        with pytest.raises(crt.CrtError, match="error -1"):
            ctx.progressive(sf.camera(), opt, crt.Sampling.make(use_gi=False), _ad(crt))
        with pytest.raises(crt.CrtError, match="error -1"):
            ctx.progressive(sf.camera(), crt.make_options(max_depth=3, shard_count=2), _smp(crt, CONFIGS[0]), _ad(crt))
        p = ctx.progressive(sf.camera(), opt, _smp(crt, CONFIGS[0]))  # a plain session takes no counts map
        p.step(1)
        a = p.arrays()
        with pytest.raises(crt.CrtError, match="error -1"):
            crt._check_core(crt.core().crtb200_accum_load_counts(ctx._h, a["sum"].ctypes.data, a["sumsq"].ctypes.data,
                                                                 a["hit0"].ctypes.data, a["counts"].ctypes.data, 1))
        pr = p.progress()
        assert pr["active_pixels"] == pr["covered_pixels"] and pr["pixel_samples"] == pr["covered_pixels"]
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
        p = ctx.progressive(sf.camera(), opt, _smp(built, cfg), _ad(built, 4, 16))
        p.run(passes_per_step=8)
        a = p.arrays()
        rgb = p.read()[0]
        p.close()
        rng = np.random.default_rng(3)
        pick = rng.integers(0, 1920 * 1080, 4096)
        ys, xs = pick // 1920, pick % 1920
        counts = a["counts"]
        assert len(np.unique(counts)) >= 3
        ps, pq = _plain_at_counts(ctx, built, sf, opt, cfg, counts)
        assert same_f32(a["sum"][ys, xs], ps[ys, xs]).all() and same_f32(a["sumsq"][ys, xs], pq[ys, xs]).all()
        assert same_f32(rgb[ys, xs], a["sum"][ys, xs] / counts[ys, xs, None].astype(np.float32)).all()
    finally:
        ctx.close()
