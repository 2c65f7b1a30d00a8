"""The sampling contract (DESIGN.md 3.10) on the CPU: the shared header's Philox, uniform and direction sampler, and the
GI oracle's images.  No GPU needed."""
import os

import numpy as np
import pytest

import gi_oracle as gio


def _unit_scene(scenes_mod, d, name, objs, materials, lights, bg=(0.2, 0.3, 0.4), w=64, h=36):
    scene = {
        "settings": {"background_color": list(bg), "width": w, "height": h, "bucket_size": 1},
        "camera": {"matrix": scenes_mod.IDENTITY, "position": [0.0, 0.0, 0.0]},
        "lights": lights, "materials": materials, "objects": objs,
    }
    scenes_mod.write_crtscene(os.path.join(d, name + ".crtscene"), scene)


@pytest.fixture(scope="module")
def unit_scenes(built, scenes_mod, tmp_path_factory):
    d = str(tmp_path_factory.mktemp("gi_scenes"))
    q = scenes_mod.quad
    diffuse = {"type": "diffuse", "albedo": [0.8, 0.6, 0.4], "smooth_shading": False}
    # one upward-facing diffuse quad under a light: every diffuse bounce escapes to the background
    _unit_scene(scenes_mod, d, "quad", [{"material_index": 0, "vertices": v, "triangles": t}
                                        for v, t in [q((-3, -1.5, -2), (3, -1.5, -2), (3, -1.5, -9), (-3, -1.5, -9))]],
                [diffuse], [{"intensity": 60, "position": [0.0, 2.0, -5.0]}])
    # a horizontal glass slab between the light and a diffuse floor
    objs = [{"material_index": 0, "vertices": v, "triangles": t}
            for v, t in [q((-6, -1.8, 1), (6, -1.8, 1), (6, -1.8, -12), (-6, -1.8, -12))]]
    objs.append({"material_index": 1, "vertices": q((-1, 0, -4), (1, 0, -4), (1, 0, -6), (-1, 0, -6))[0],
                 "triangles": q((-1, 0, -4), (1, 0, -4), (1, 0, -6), (-1, 0, -6))[1]})
    _unit_scene(scenes_mod, d, "glass", objs, [diffuse, {"type": "refractive", "albedo": None, "ior": 1.5, "smooth_shading": False}],
                [{"intensity": 90, "position": [0.0, 3.0, -5.0]}], bg=(0.0, 0.0, 0.0))
    out = {}
    for name in ("quad", "glass"):
        sf = built.SceneFile(name + ".crtscene", d)
        out[name] = (sf, sf.flatten())
    return out


def test_philox_known_answers():
    assert gio.philox([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert gio.philox([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_unit_range():
    assert gio.unit(0) == 0.0
    assert gio.unit(0xFFFFFFFF) == np.float32(1 - 2.0 ** -24)
    assert gio.unit(0x80000000) == 0.5


def _normals():
    rng = np.random.default_rng(7)
    n = rng.normal(size=(200, 3))
    n = (n / np.linalg.norm(n, axis=1, keepdims=True)).astype(np.float32)
    special = np.array([[0, 0, 1], [0, 0, -1], [0, 0, -0.0], [1, 0, 0], [0, -1, 0]], np.float32)
    special[2] = [0.0, 0.0, -0.0]
    return np.concatenate([special, n])


def test_tangent_frame_orthonormal():
    for n in _normals():
        if not np.any(n):  # (0, 0, -0.0): the frame is still defined (negative branch)
            t, b = gio.tangent_frame(n)
            assert np.all(np.isfinite(t)) and np.all(np.isfinite(b))
            continue
        t, b = gio.tangent_frame(n)
        m = np.stack([t, b, n]).astype(np.float64)
        assert np.allclose(m @ m.T, np.eye(3), atol=1e-6), (n, t, b)


def test_direction_sampler_statistics():
    n = np.array([0.3, -0.5, 0.8], np.float32)
    n = (n / np.linalg.norm(n)).astype(np.float32)
    d = gio.diffuse_dirs(n, 1_000_000, seed=3, frame=1, p=12345, s=2, key0=0, k=0).astype(np.float64)
    cos = d @ n.astype(np.float64)
    assert np.all(cos > 0)
    assert np.max(np.abs(np.linalg.norm(d, axis=1) - 1.0)) < 4 * 2.0 ** -23
    sigma = np.sqrt(1.0 / 18.0 / len(cos))  # cosine-weighted: E[cos] = 2/3, Var[cos] = 1/2 - 4/9
    assert abs(cos.mean() - 2.0 / 3.0) < 4 * sigma
    # nan normal -> nan direction
    assert np.all(np.isnan(gio.diffuse_dirs(np.array([np.nan, 0, 1], np.float32), 1)))


def _opts(built, depth):
    return built.make_options(max_depth=depth)


def test_oracle_thread_count_invariant(built, loaded):
    sf, flat, rects, n = loaded["hw11_room"]
    opt = built.make_options(max_depth=3, rects=rects, n_rects=n)
    smp = built.Sampling.make(gi_samples=2, rays_per_pixel=2, seed=5)
    a, ha, sa = gio.render_sampled(flat, sf.camera(), opt, smp, threads=1)
    b, hb, sb = gio.render_sampled(flat, sf.camera(), opt, smp, threads=16)
    assert a.tobytes() == b.tobytes() and ha.tobytes() == hb.tobytes() and sa == sb
    assert sa["rays_diffuse"] > 0


def test_exact_identity_escaping_bounces(built, unit_scenes):
    sf, flat = unit_scenes["quad"]
    opt = _opts(built, 3)
    base = np.float32([0.8, 0.6, 0.4])
    bg = np.float32([0.2, 0.3, 0.4])
    img0, hits, _ = gio.render_sampled(flat, sf.camera(), opt, built.Sampling.make(gi_samples=0, seed=9))
    on = hits["mesh"] >= 0
    assert on.sum() > 100 and (~on).sum() > 100
    for G in (1, 2, 5):
        img, _, st = gio.render_sampled(flat, sf.camera(), opt, built.Sampling.make(gi_samples=G, seed=9))
        S = np.zeros(3, np.float32)
        for _ in range(G):
            S = (S + bg).astype(np.float32)
        want = np.where(on[..., None], ((img0 + base * S).astype(np.float32) / np.float32(G + 1)).astype(np.float32), img0)
        assert img.tobytes() == want.astype(np.float32).tobytes(), G
        assert st["rays_diffuse"] == G * int(on.sum())


def test_refractive_meshes_cast_shadows_with_gi(built, ob, unit_scenes):
    sf, flat = unit_scenes["glass"]
    opt = _opts(built, 2)
    h, w = sf.info.height, sf.info.width
    row, col = int(0.68 * h), w // 2  # floor point (0, -1.8, -5), under the slab
    off, _, _ = ob.render(flat, sf.camera(), opt)
    on, _, _ = gio.render_sampled(flat, sf.camera(), opt, built.Sampling.make(gi_samples=0))
    assert np.all(off[row, col] > 0), off[row, col]
    assert np.all(on[row, col] == 0), on[row, col]
