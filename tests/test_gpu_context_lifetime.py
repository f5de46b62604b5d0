"""-m gpu: a context owns its device buffers.  Closing it (rrtb_destroy) gives back everything it allocated -- the scene
and build arrays, the accumulator and framebuffer of the host render path, the multi-GPU frame -- so an application
that opens and closes contexts does not grow on the device."""
import os

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

W = H = 8192
# Device memory one cycle's context allocates: the 64-bit accumulator and the framebuffer (room for doubles) of rrtb_render,
# the frame and the 64-bit sum buffer of rrtb_frame_create, 3*W*H words of 8 bytes each (6.4 GB).  The scene's arrays
# are small beside them.
CONTEXT_BYTES = 4 * 3 * W * H * 8


def _free_bytes():
    import torch

    torch.cuda.synchronize(0)
    return torch.cuda.mem_get_info(0)[0]


def _cycle(inside=lambda: None):
    from rrt_b200 import Context, Scene

    with Context(0) as ctx:
        ctx.set_scene(Scene.from_file(os.path.join(ROOT, "tests", "golden", "scenes", "final.txt"), W, H))
        ctx.render(W, H, 1, 1, seed=7)  # the 0.8 GB host copy is dropped at once
        ctx.frame_create(W, H)
        inside()


def test_close_gives_back_the_device_memory():
    # the first cycle loads the modules and whatever else the CUDA runtime allocates lazily, once per process
    _cycle()
    base = _free_bytes()
    # other work may share the card: the margins are half of what the context allocates
    for k in range(3):

        def inside():
            used = base - _free_bytes()
            assert used >= CONTEXT_BYTES // 2, (k, used, CONTEXT_BYTES)  # the measurement sees the context's buffers

        _cycle(inside)
        left = base - _free_bytes()
        assert abs(left) <= CONTEXT_BYTES // 2, (k, left, CONTEXT_BYTES)
