"""Progressive sessions (DESIGN.md 3.10.1) on the CPU: the restatement's accumulator entry point agrees with its one-shot
image, and the Python session API goes to the CUDA core with no CPU fallback.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest

import gi_oracle as gio
import progressive_oracle as po
from conftest import same_f32


@pytest.mark.parametrize("name", ["hw11_room", "hw12_textures", "degenerate_uv", "uncovered"])
def test_sums_divide_to_the_sampled_image(name, loaded, crt):
    sf, flat, rects, n = loaded[name]
    opt = crt.make_options(max_depth=3, rects=rects, n_rects=n)
    smp = crt.Sampling.make(gi_samples=1, rays_per_pixel=3, seed=5)
    s, q = po.render_sums(flat, sf.camera(), opt, smp)
    rgb, _, _ = gio.render_sampled(flat, sf.camera(), opt, smp, want_hits=False)
    assert same_f32(s / np.float32(3), rgb).all()
    assert not (q < 0).any()  # (degenerate_uv has NaN pixels)


def test_one_sample_sumsq_is_the_square(loaded, crt):
    sf, flat, rects, n = loaded["hw11_room"]
    opt = crt.make_options(max_depth=5, rects=rects, n_rects=n)
    s, q = po.render_sums(flat, sf.camera(), opt, crt.Sampling.make(gi_samples=2, rays_per_pixel=1, seed=9))
    assert same_f32(q, s * s).all()
    assert s.any()


def test_progressive_has_no_cpu_fallback(built, loaded, tmp_path):
    """Without a usable sm_100 device a progressive session fails loudly instead of rendering on the CPU."""
    n = C.c_int(-1)
    rc = built.core().crtb200_device_count(C.byref(n))
    if rc == 0 and n.value > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(built.CrtError):
        built.Context(0)
    # a context that never reached a device (no handle): every session call must still go to the CUDA core and fail
    sf, flat, rects, nr = loaded["hw11_room"]
    ctx = object.__new__(built.Context)
    ctx._h = C.c_void_p()
    ctx.width, ctx.height, ctx._session = sf.info.width, sf.info.height, None
    cam, opt, smp = sf.camera(), built.make_options(max_depth=3, rects=rects, n_rects=nr), built.Sampling.make(seed=1)
    with pytest.raises(built.CrtError):
        ctx.progressive(cam, opt, smp)
    h, w = ctx.height, ctx.width
    path = str(tmp_path / "s.npz")
    np.savez(path, sum=np.zeros((h, w, 3), np.float32), sumsq=np.zeros((h, w, 3), np.float32),
             hit0=np.zeros((h, w), built.HIT_DTYPE), samples=np.uint32(1), **built._session_params(w, h, cam, opt, smp))
    with pytest.raises(built.CrtError):
        ctx.resume(path, cam, opt, smp)
