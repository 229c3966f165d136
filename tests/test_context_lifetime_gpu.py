"""Destroying a context while work is still enqueued on every stream it owns, the lazily made ones included (band DMA,
ordered flag writes, mesh build graph, pipelined presentation): ore_destroy waits for that work, writes the
ORE_DEBUG_BLOCK_CYCLES dump in its documented layout and frees everything, and a fresh context renders as before."""
import numpy as np
import pytest

from test_mesh_refit_cpu import torus_arrays

pytestmark = pytest.mark.gpu


def test_destroy_with_work_in_flight(pkg, tmp_path, monkeypatch):
    import torch
    F = pkg.capi
    W, H = 160, 96
    sc = pkg.scene.reference_scene(64, 3)
    cams = [pkg.scene.reference_camera(), pkg.scene.orbit_camera(sc, 40), pkg.scene.orbit_camera(sc, 120)]
    dump = tmp_path / "block_cycles.bin"
    monkeypatch.setenv("ORE_DEBUG_BLOCK_CYCLES", str(dump))
    r = pkg.Renderer(0)
    monkeypatch.delenv("ORE_DEBUG_BLOCK_CYCLES")
    r.set_scene(sc)
    want = torch.zeros((len(cams), H, W), dtype=torch.int32, device="cuda:0")
    for i, cam in enumerate(cams):
        r.render_device(cam, W, H, want[i].data_ptr())
    # band DMA: the band stream and its events
    band = torch.full((2, H, W), 0x5A5A5A5A, dtype=torch.int32, device="cuda:0")
    r.render_batch_device(cams[1:], W, H, [band[0].data_ptr(), band[1].data_ptr()], out_pitch=W, flags=F.ORE_FLAG_BAND_DMA)
    # ordered flag write: the signal stream and its events (no signal stream before the first one)
    flag = torch.zeros(64, dtype=torch.int32, device="cuda:0")
    assert r.stream_handle(2) == 0
    r.flag_write_after(flag.data_ptr(), 7)
    assert r.stream_handle(2) != 0
    # device mesh build: the capture stream and the graph
    tris = torch.from_numpy(np.ascontiguousarray(torus_arrays()[0], np.float32)).to("cuda:0")
    r.set_mesh_device(tris, True)
    # pipelined presentation: the copy stream
    shown = np.zeros((H, W), dtype=np.uint32)
    r.render_async(cams[0], W, H, out=shown)
    r.close()   # no wait(): the work above may still be enqueued

    raw = dump.read_bytes()
    cap = int(np.frombuffer(raw[:8], dtype=np.uint64)[0])
    assert cap > 0 and len(raw) == 8 + 4 * 2 * cap, (cap, len(raw))
    assert np.frombuffer(raw[8:], dtype=np.uint32).any()
    torch.cuda.synchronize()
    assert int(flag[0]) == 7
    assert torch.equal(band, want[1:])
    assert shown.any()

    fresh = pkg.Renderer(0)
    try:
        fresh.set_scene(sc)
        got = torch.zeros((H, W), dtype=torch.int32, device="cuda:0")
        fresh.render_device(cams[0], W, H, got.data_ptr())
        fresh.synchronize()
        assert torch.equal(got, want[0])
    finally:
        fresh.close()
