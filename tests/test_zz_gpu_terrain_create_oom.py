"""rvb_terrain_create when the device cannot hold the layer: the call fails with RVB_ERR_CUDA, returns no handle, and leaves
nothing behind that fails the next call -- neither the next layer's build nor the caller's own CUDA work."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

RVB_ERR_CUDA = -2


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import isaac_rover_b200
    return isaac_rover_b200


def test_terrain_create_fails_cleanly_when_the_index_copy_does_not_fit(R):
    w = R.synth.make_world(length=20.0, nv=72, K=200, n_stones=12, seed=1)
    lib = R._lib.load()
    tri = w.triangles.to("cuda:0", torch.int32).contiguous()
    ver = w.vertices.to("cuda:0", torch.float16).contiguous()
    # a [G,G,K] index whose K-contiguous copy would take 4 * G * G * K = 4.4 TB: more than any device holds, so the first
    # allocation of the build fails and nothing is reserved.  All strides 0: the call never gets far enough to read it.
    G, K = 1 << 14, 4096
    idx = torch.zeros(1, 1, 1, dtype=torch.int32, device="cuda:0").expand(G, G, K)
    h = C.c_void_p(1)
    rc = lib.rvb_terrain_create(C.byref(h), R._lib.ptr(idx), G, G, K, 0, 0, 0, R._lib.ptr(tri), tri.shape[0], R._lib.ptr(ver),
                                ver.shape[0], 0.1, 0.0, 0.0, R.SEM_TORCH_CUDA, 0, R._lib.stream_of(idx))
    assert rc == RVB_ERR_CUDA
    assert h.value is None
    assert "cudaMalloc" in lib.rvb_last_error().decode()
    # the next valid layer builds, block and superblock lists included (K = 200 <= 255), and torch's own launches still succeed
    layer = R.TerrainLayer(w.map_indices, w.triangles, w.vertices, torch.tensor([0, 0, 0.0]))
    assert layer.has_index and layer.bytes() > 0
    assert int(torch.arange(10, device="cuda:0").sum()) == 45
    layer.close()
