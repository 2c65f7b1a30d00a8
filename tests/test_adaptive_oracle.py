"""Adaptive progressive sessions (DESIGN.md 3.10.2) on the CPU: known answers of the shared stop rule, the restatement's
per-pixel prefix property, and the new entry points going to the CUDA core with no CPU fallback.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest

import adaptive_oracle as ao
import progressive_oracle as po
from conftest import same_f32


def _rule(n, S, Q, mn, mx, ae, re):
    """The stop rule, written out in numpy float32 in the order crt_sampling.h gives."""
    f = np.float32
    if n >= mx:
        return True
    if n < mn:
        return False
    nf = f(n)
    for c in range(3):
        m = f(S[c]) / nf
        v = (f(Q[c]) - f(S[c]) * m) / (nf - f(1))
        v = v if v > 0 else f(0)
        e = np.sqrt(v / nf, dtype=np.float32)
        tol = f(ae) + f(re) * abs(m)
        if not e <= tol:
            return False
    return True


def test_stop_rule_known_answers(crt):
    ad = crt.Adaptive.make(min_samples=4, max_samples=16, abs_error=0.01, rel_error=0.05)
    flat = ([2.0, 2.0, 2.0], [1.0, 1.0, 1.0])  # c = 0.5 every sample: zero variance
    assert not ao.adapt_stop(3, [1.5] * 3, [0.75] * 3, ad)  # below min_samples
    assert ao.adapt_stop(4, *flat, ad)  # zero variance stops at min_samples
    nan = ([np.nan, 1.0, 1.0], [np.nan, 1.0, 1.0])
    for n in (4, 8, 15):
        assert not ao.adapt_stop(n, *nan, ad)  # a NaN mean never stops early
    assert ao.adapt_stop(16, *nan, ad)  # ... but max_samples caps it
    assert ao.adapt_stop(16, [0.0, 100.0, 3.0], [0.0, 1e6, 9.0], ad)  # the cap, whatever the noise
    big = ([1e6, 1e6, 1e6], [3e38, 3e38, 3e38])  # large Q: a large variance, no stop below the cap
    assert not ao.adapt_stop(8, *big, ad)
    rng = np.random.default_rng(7)
    for _ in range(400):
        n = int(rng.integers(1, 20))
        c = rng.random((n, 3)).astype(np.float32) * np.float32(rng.choice([0.01, 0.5, 4.0]))
        S = np.zeros(3, np.float32)
        Q = np.zeros(3, np.float32)
        for x in c:
            S = S + x
            Q = Q + x * x
        a = crt.Adaptive.make(min_samples=int(rng.integers(2, 8)), max_samples=18, abs_error=float(rng.choice([0, 0.02, 0.2])),
                              rel_error=float(rng.choice([0, 0.1])))
        assert ao.adapt_stop(n, S, Q, a) == _rule(n, S, Q, a.min_samples, a.max_samples, a.abs_error, a.rel_error)


@pytest.mark.parametrize("name", ["hw11_room", "hw12_textures", "degenerate_uv", "uncovered"])
def test_adaptive_sums_are_prefix_sums(name, loaded, crt):
    sf, flat, rects, nr = loaded[name]
    opt = crt.make_options(max_depth=3, rects=rects, n_rects=nr)
    smp = crt.Sampling.make(gi_samples=1, seed=5)
    ad = crt.Adaptive.make(min_samples=2, max_samples=6, abs_error=0.02, rel_error=0.05)
    s, q, counts, _ = ao.render_adaptive(flat, sf.camera(), opt, smp, ad, passes=7)
    assert counts.max() <= 6
    for n in np.unique(counts):
        if n == 0:
            continue
        smp.rays_per_pixel = int(n)
        ps, pq = po.render_sums(flat, sf.camera(), opt, smp)
        m = counts == n
        assert same_f32(s[m], ps[m]).all() and same_f32(q[m], pq[m]).all(), (name, n)


def test_adaptive_abi_has_no_cpu_fallback(built, loaded):
    """Every adaptive entry point exists in the CUDA core and fails without a device instead of rendering on the CPU."""
    lib = built.core()
    n = C.c_int(-1)
    rc = lib.crtb200_device_count(C.byref(n))
    if rc == 0 and n.value > 0:
        pytest.skip("a GPU is present")
    for fn in ("crtb200_accum_begin_adaptive", "crtb200_accum_progress", "crtb200_accum_counts", "crtb200_accum_load_counts"):
        assert hasattr(lib, fn), fn
    sf, flat, rects, nr = loaded["hw11_room"]
    ctx = object.__new__(built.Context)
    ctx._h = C.c_void_p()
    ctx.width, ctx.height, ctx._session = sf.info.width, sf.info.height, None
    cam, opt, smp = sf.camera(), built.make_options(max_depth=3, rects=rects, n_rects=nr), built.Sampling.make(seed=1)
    with pytest.raises(built.CrtError):
        ctx.progressive(cam, opt, smp, built.Adaptive.make())
    for rc in (lib.crtb200_accum_progress(None, C.byref(built.AccumProgress())), lib.crtb200_accum_counts(None, None),
               lib.crtb200_accum_load_counts(None, None, None, None, None, 0)):
        assert rc != 0
