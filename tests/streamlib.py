"""Helpers of the stream-ordered update tests (ore_set_spheres_device, ore_set_mesh_device,
ore_set_mesh_triangles_device): a stream held by a host flag, and the "rejected and unchanged" check."""
import threading
import time

import numpy as np


def _held_stream(renderer, update, after=None):
    """enqueues `update` on a stream held by a host flag; returns (seconds the call took, still pending at return);
    `after` runs while the stream is still held"""
    import torch
    flag = renderer.host_alloc((16,))
    flag[:] = 0
    S = torch.cuda.Stream()
    timer = threading.Timer(2.0, lambda: flag.__setitem__(0, 1))   # releases the stream in every case
    try:
        torch.cuda.synchronize()
        renderer.flag_wait_geq(flag.ctypes.data, 1, S.cuda_stream)
        timer.start()
        t0 = time.perf_counter()
        update(S.cuda_stream)
        dt = time.perf_counter() - t0
        pending = not S.query()
        if after is not None:
            after()
        timer.join()
        S.synchronize()
        return dt, pending
    finally:
        timer.cancel()
        flag[0] = 1
        torch.cuda.synchronize()
        renderer.synchronize()
        renderer.host_free(flag)


def assert_rejected(call, bad, render, want):
    """call(*args) returns ORE_ERR_INVALID (1) for every argument tuple of `bad`, and render() still gives `want`"""
    for args in bad:
        rc = call(*args)
        assert rc == 1, (args, rc)
        assert np.array_equal(render(), want), args
