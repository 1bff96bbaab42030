"""A context's buffers across state changes (-m gpu): batches, asynchronous batches, resolution changes, the number of frames in
flight, a caller's stream and an external framebuffer, one after another on the same context. Every frame and raybuffer equals a
single cvx_draw of the same setup at the same resolution on a separate context."""
from __future__ import annotations

import numpy as np
import pytest

from conftest import POSES, setup_for

pytestmark = pytest.mark.gpu

BIG, SMALL = (333, 217), (160, 96)


@pytest.fixture(scope="module")
def single(cv, mill_world):
    """(W, H, pose index) -> (frame, td, lr) of one cvx_draw into raybuffers cleared to 0, on a context of its own."""
    rm = cv.RenderManager(0)
    rm.upload_world(mill_world)
    cache = {}

    def get(W, H, i):
        if (W, H, i) not in cache:
            rm.set_resolution(W, H)
            rm.clear_raybuffers(0)
            rm.draw_setup(setup_for(cv, mill_world, POSES[i], W, H))
            rm.sync()
            cache[W, H, i] = (rm.read_frame(), *rm.read_raybuffers())
        return cache[W, H, i]

    yield get
    rm.destroy()


@pytest.fixture
def rm(cv, mill_world):
    m = cv.RenderManager(0)
    m.upload_world(mill_world)
    yield m
    m.destroy()


class _DeviceWords:
    """`n` int32 words at a device address, for torch.as_tensor."""
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False), "strides": None, "version": 2}


def _device_frame(rm):
    import torch
    rm.sync()
    ptr, nbytes = rm.device_frame_ptr()
    return torch.as_tensor(_DeviceWords(ptr, nbytes // 4), device="cuda:0").cpu().numpy().view(np.uint32).reshape(rm.height, rm.width)


def _setups(cv, world, views, W, H):
    return [setup_for(cv, world, POSES[i], W, H) for i in views]


def _check_frames(single, dst, views, W, H, what):
    for k, i in enumerate(views):
        assert np.array_equal(dst[k], single(W, H, i)[0]), (what, k)


def _check_last_view(rm, single, i, what, raybuffers=True):
    frame, td, lr = single(rm.width, rm.height, i)
    assert np.array_equal(rm.read_frame(), frame), what
    assert np.array_equal(_device_frame(rm), frame), what
    if raybuffers:
        got_td, got_lr = rm.read_raybuffers()
        assert np.array_equal(got_td, td) and np.array_equal(got_lr, lr), what


def _pinned(cv, n, W, H):
    d = cv.alloc_pinned((n, H, W))
    d[:] = 0
    return d


def test_batches_across_resolution_changes(cv, rm, mill_world, single):
    """Each resolution change reallocates every slot: the last view's frame and raybuffers (views <= slots, so that slot held only that
    view since its allocation) are what the read functions and the device pointer return."""
    rm.set_frames_in_flight(6)
    for (W, H), views in ((BIG, range(0, 6)), (SMALL, range(6, 10)), (BIG, range(2, 7))):
        rm.set_resolution(W, H)
        dst = _pinned(cv, len(views), W, H)
        rm.draw_batch(_setups(cv, mill_world, views, W, H), dst)
        _check_frames(single, dst, views, W, H, (W, H))
        _check_last_view(rm, single, views[-1], (W, H))
        cv.native.lib.cvx_free_pinned(dst.ctypes.data)


def test_frames_in_flight_grow_then_shrink(cv, rm, mill_world, single):
    W, H = BIG
    rm.set_resolution(W, H)
    views = [(3 * j) % len(POSES) for j in range(11)]
    setups = _setups(cv, mill_world, views, W, H)
    dst = _pinned(cv, len(views), W, H)
    for k in (8, 2):
        rm.set_frames_in_flight(k)
        dst[:] = 0
        rm.draw_batch(setups, dst)
        _check_frames(single, dst, views, W, H, k)
        _check_last_view(rm, single, views[-1], k, raybuffers=False)
    cv.native.lib.cvx_free_pinned(dst.ctypes.data)


def test_resolution_change_behind_an_asynchronous_batch(cv, rm, mill_world, single):
    W, H = BIG
    rm.set_resolution(W, H)
    views = list(range(len(POSES)))
    dst = _pinned(cv, len(views), W, H)
    b = rm.draw_batch_async(_setups(cv, mill_world, views, W, H), dst)
    rm.set_resolution(*SMALL)
    rm.batch_wait(b)
    _check_frames(single, dst, views, W, H, "async before resize")
    small = _pinned(cv, 4, *SMALL)
    rm.draw_batch(_setups(cv, mill_world, range(4), *SMALL), small)
    _check_frames(single, small, range(4), *SMALL, "after resize")
    _check_last_view(rm, single, 3, "after resize")
    for d in (dst, small):
        cv.native.lib.cvx_free_pinned(d.ctypes.data)


def test_batches_on_a_caller_stream_then_the_own_stream(cv, rm, mill_world, single):
    import torch
    W, H = BIG
    rm.set_resolution(W, H)
    views = [1, 4, 7, 0, 9, 5, 2, 8]
    setups = _setups(cv, mill_world, views, W, H)
    dsts = [_pinned(cv, len(views), W, H) for _ in range(3)]
    stream = torch.cuda.Stream(device=0)
    rm.set_stream(stream.cuda_stream)
    rm.draw_batch(setups, dsts[0])
    b = rm.draw_batch_async(setups[::-1], dsts[1])
    rm.batch_wait(b)
    _check_frames(single, dsts[0], views, W, H, "caller stream")
    _check_frames(single, dsts[1], views[::-1], W, H, "caller stream, async")
    _check_last_view(rm, single, views[0], "caller stream, async", raybuffers=False)
    rm.set_stream(0)
    rm.draw_batch(setups, dsts[2])
    _check_frames(single, dsts[2], views, W, H, "own stream")
    _check_last_view(rm, single, views[-1], "own stream", raybuffers=False)
    for d in dsts:
        cv.native.lib.cvx_free_pinned(d.ctypes.data)


def test_batch_into_an_external_frame(cv, rm, mill_world, single):
    import torch
    W, H = BIG
    rm.set_resolution(W, H)
    views = [6, 2, 9]
    external = torch.zeros(H * W, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    rm.set_external_frame(external.data_ptr())
    dst = _pinned(cv, len(views), W, H)
    rm.draw_batch(_setups(cv, mill_world, views, W, H), dst)
    _check_frames(single, dst, views, W, H, "external")
    rm.sync()
    last = single(W, H, views[-1])
    assert np.array_equal(external.cpu().numpy().view(np.uint32).reshape(H, W), last[0])
    _check_last_view(rm, single, views[-1], "external", raybuffers=False)
    rm.set_external_frame(0)
    cv.native.lib.cvx_free_pinned(dst.ctypes.data)
