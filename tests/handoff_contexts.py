"""TEST INFRASTRUCTURE ONLY.  Contexts whose tail hand-off to k_coop (DESIGN.md 3.8) is forced or switched off through the
tuning environment that context creation reads once per GPU (crtb200_create and crtb200_create_multi read it for every
GPU of their list, so all GPUs of a multi-GPU context get the same settings)."""
import os

# every walk still running once the queue is dry (a small frame's queue is dry after the first refill) is handed off
# before its next step, with room for all of them
_ALL = dict(CRT_TAIL_ITERS=0, CRT_TAIL_START=0, CRT_TAIL_SMALL=100000000, CRT_TAIL_CAP=1000000)
HANDOFF_ENV = {
    "default": {},                                     # the shipped policy
    "all": _ALL,                                       # k_coop does all the traversal work of the frame
    "mid": dict(_ALL, CRT_TAIL_ITERS=3, CRT_TAIL_START=3),  # walks that took 3 node-phase iterations: mid-flight records
    "final_only": dict(_ALL, CRT_COOP_EARLY=0),        # as "all", with k_coop's early pass switched off
    "off": dict(CRT_TAIL_ITERS=-1),                    # no hand-off
    # as "all", with the smallest capacity crtb200_create accepts (1 walk per resident k_coop warp): once it is used up,
    # the lanes that still ask keep walking in the traversal kernel
    "capped": dict(_ALL, CRT_TAIL_CAP=1),
}
HANDOFF = list(HANDOFF_ENV)


def ctx_with_env(crt, devices=0, **env):
    """A Context (one device index or a list of them) created under tuning environment variables."""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return crt.Context(devices)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


def handoff_context(crt, which, devices=0):
    return ctx_with_env(crt, devices, **HANDOFF_ENV[which])


class HandoffContexts:
    """handoff_context per (name, device list), created on first use and closed together (a module fixture's)."""

    def __init__(self, crt):
        self._crt = crt
        self._ctx = {}

    def __call__(self, which, devices=0):
        key = (which, tuple(devices) if isinstance(devices, (list, tuple)) else devices)
        if key not in self._ctx:
            self._ctx[key] = handoff_context(self._crt, which, devices)
        return self._ctx[key]

    def close(self):
        for ctx in self._ctx.values():
            ctx.close()
        self._ctx.clear()
