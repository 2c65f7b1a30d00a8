"""Progressive-session calls that render nothing (read, save, counts, progress, resume; DESIGN.md 3.10.1 / 3.10.2)
leave the context's last render alone, keep the per-pixel counts of plain sessions, and store only the session's
pixels."""
import numpy as np
import pytest

from conftest import same_f32
from test_gpu_progressive import _context, _covered, _oneshot, _same_frame, _smp

pytestmark = pytest.mark.gpu
DEVICES = pytest.mark.parametrize("devices", [0, [0, 0, 0]], ids=["single", "multi"])
CFG = dict(G=1, depth=5)


def _options(crt, loaded, name, depth=CFG["depth"]):
    sf, flat, rects, n = loaded[name]
    return sf, flat, crt.make_options(max_depth=depth, rects=rects, n_rects=n), _covered((sf.info.height, sf.info.width), rects, n)


@DEVICES
@pytest.mark.parametrize("adaptive", [False, True], ids=["plain", "adaptive"])
def test_calls_keep_last_render_stats(devices, adaptive, loaded, crt, tmp_path):
    sf, flat, opt, _ = _options(crt, loaded, "uncovered")
    ad = crt.Adaptive.make(min_samples=2, max_samples=6, abs_error=0.01, rel_error=0.03) if adaptive else None
    path = str(tmp_path / "session.npz")
    ctx = _context(crt, sf, flat, devices)
    try:
        p = ctx.progressive(sf.camera(), opt, _smp(crt, CFG), ad)

        def unchanged(p):
            before = (ctx.last_stats(), ctx.sampling_stats())
            p.read(want_rgb8=True, want_hits=True)
            p.arrays()
            p.progress()
            p.save(path)
            p = ctx.resume(path, sf.camera(), opt, _smp(crt, CFG), ad)
            p.read()
            assert (ctx.last_stats(), ctx.sampling_stats()) == before
            return p

        p.step(3)
        p = unchanged(p)
        # a one-shot render of another sampling, depth and coverage
        ctx.set_sampling(crt.Sampling.make(gi_samples=3, rays_per_pixel=2, seed=5))
        ctx.render(sf.camera(), crt.make_options(max_depth=2))
        ctx.set_sampling(None)
        assert ctx.sampling_stats()["samples"] == 2
        unchanged(p)
    finally:
        ctx.close()


@DEVICES
def test_plain_counts_follow_rects(devices, loaded, crt, tmp_path):
    sf, flat, opt, cov = _options(crt, loaded, "uncovered")
    assert not cov.all()
    path = str(tmp_path / "session.npz")
    ctx = _context(crt, sf, flat, devices)
    try:
        p = ctx.progressive(sf.camera(), opt, _smp(crt, CFG))
        assert np.array_equal(p.counts(), np.zeros(cov.shape, np.uint32))
        p.step(1)
        p.step(3)
        assert np.array_equal(p.counts(), np.where(cov, 4, 0).astype(np.uint32))
        assert p.progress()["covered_pixels"] == cov.sum()
        p.save(path)
        p = ctx.resume(path, sf.camera(), opt, _smp(crt, CFG))
        assert np.array_equal(p.counts(), np.where(cov, 4, 0).astype(np.uint32))
        p.step(2)
        assert np.array_equal(p.counts(), np.where(cov, 6, 0).astype(np.uint32))
        assert p.progress() == dict(passes=6, covered_pixels=cov.sum(), active_pixels=cov.sum(), pixel_samples=6 * cov.sum())
    finally:
        ctx.close()


@DEVICES
def test_read_keeps_uncovered_pixels(devices, loaded, crt):
    sf, flat, opt, cov = _options(crt, loaded, "uncovered")
    ctx = _context(crt, sf, flat, devices)
    try:
        p = ctx.progressive(sf.camera(), opt, _smp(crt, CFG))
        p.step(2)
        full = _oneshot(ctx, crt, sf, dict(G=2, depth=3), 3, crt.make_options(max_depth=3), seed=4)
        rgb, rgb8, hits = p.read(want_rgb8=True, want_hits=True)
        assert same_f32(rgb[~cov], full[0][~cov]).all() and np.array_equal(rgb8[~cov], full[1][~cov])
        assert (hits["mesh"][~cov] == -1).all() and (hits["triangle"][~cov] == -1).all()
        _same_frame((rgb, rgb8, hits), _oneshot(ctx, crt, sf, CFG, 2, opt), np.ones(cov.shape, bool))
    finally:
        ctx.close()


@DEVICES
def test_read_after_render_of_other_gi_samples(devices, loaded, crt):
    sf, flat, opt, cov = _options(crt, loaded, "hw11_room")
    ctx = _context(crt, sf, flat, devices)
    try:
        p = ctx.progressive(sf.camera(), opt, _smp(crt, CFG))
        p.step(4)
        _oneshot(ctx, crt, sf, dict(G=4, depth=4), 1, crt.make_options(max_depth=4))
        got = p.read(want_rgb8=True, want_hits=True)
        _same_frame(got, _oneshot(ctx, crt, sf, CFG, 4, opt), cov)
    finally:
        ctx.close()
