"""Closing a context (crtb200_destroy) frees everything it created: its buffers, streams and events, including those
made on first use by host-bound frames, frame batches, device frames, progressive sessions, ray queries and device tree
builds, and after a call that failed its checks.  Closing twice is harmless, repeated cycles give the device's memory
back, and a context made afterwards renders what the first one did."""
import os

import pytest

pytestmark = pytest.mark.gpu
DEVICES = pytest.mark.parametrize("devices", [0, [0, 0, 0]], ids=["single", "multi"])
CYCLES = 5
MAX_LOSS = 256 << 20      # free memory the cycles may lose overall (other work can share the GPU)
QUEUE_BUDGET = 4 << 30    # per GPU of a context: the GI step below plans its queues up to it


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def room(built, scenes_mod, tmp_path_factory):
    """hw11_room at 1280x720: a host-bound frame of this size plans two chunk streams and the band stream"""
    d = str(tmp_path_factory.mktemp("lifecycle"))
    scenes_mod.write_crtscene(os.path.join(d, "room.crtscene"), scenes_mod.hw11_room(width=1280, height=720, sphere_n=8))
    sf = built.SceneFile("room.crtscene", d)
    return sf, sf.flatten(trees=False)


def _free(torch):
    """the device's free memory after a synchronise: the best of three reads"""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return max(torch.cuda.mem_get_info(0)[0] for _ in range(3))


def _cycle(crt, torch, sf, geo, devices):
    """One context through every resource it creates on first use, closed twice.  Returns its host-bound frame and the
    free memory read while it was open."""
    cam = sf.camera()
    dev = torch.device("cuda", 0)
    ctx = crt.Context(devices)
    ctx.set_queue_budget(QUEUE_BUDGET)
    ctx.upload_geometry(geo, keepalive=sf)  # keeps the built trees
    opt = crt.make_options(max_depth=5)
    frame = ctx.render(cam, opt, want_rgb=True, want_rgb8=True, want_hits=True)[:3]
    # two frames: the copy stream, the second frame pair, and the swap of the pairs
    ctx.render_frames([sf.camera(), crt.camera_pan(sf.camera(), 5.0)], opt, want_rgb8=True)
    d_rgb = torch.empty((ctx.height, ctx.width, 3), dtype=torch.float32, device=dev)
    ctx.render_device(cam, opt, d_rgb=d_rgb.data_ptr(), stream=torch.cuda.current_stream(dev).cuda_stream)
    ctx.last_stats()
    # an adaptive session left open; gi_samples 4 at depth 4 plans the queues up to the budget
    p = ctx.progressive(cam, crt.make_options(max_depth=4), crt.Sampling.make(gi_samples=4, seed=3),
                        crt.Adaptive.make(min_samples=2, max_samples=8))
    p.step(2)
    rays = ctx.generate_rays_device(cam)
    ctx.trace(rays, crt.RAY_PRIMARY)
    ctx.trace(rays, crt.RAY_SHADOW, max_distance=torch.full(rays.shape[:-1], 2.0, device=dev))
    ctx.query_stats()
    with pytest.raises(crt.CrtError):
        ctx.render(cam, crt.make_options(max_depth=32))
    del d_rgb, rays
    held = _free(torch)
    ctx.close()
    ctx.close()
    return frame, held


@DEVICES
def test_close_frees_everything(devices, room, built, torch):
    sf, geo = room
    before = _free(torch)
    frames = []
    for _ in range(CYCLES):
        frame, held = _cycle(built, torch, sf, geo, devices)
        assert before - held >= 10 * MAX_LOSS, f"the open context held only {(before - held) >> 20} MiB"
        frames.append(frame)
    after = _free(torch)
    assert before - after < MAX_LOSS, f"{CYCLES} cycles lost {(before - after) >> 20} MiB of device memory"

    ctx = built.Context(devices)
    try:
        ctx.upload_geometry(geo, keepalive=sf)
        again = ctx.render(sf.camera(), built.make_options(max_depth=5), want_rgb=True, want_rgb8=True, want_hits=True)[:3]
    finally:
        ctx.close()
    for name, a, b in zip(("rgb", "rgb8", "hits"), frames[0], again):
        assert a.tobytes() == b.tobytes(), f"{name} of a fresh context differs from the first cycle's"
