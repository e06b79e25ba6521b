"""Terrain-layer handle (index + mesh of one layer) around rvb_terrain_create/destroy."""
import ctypes as C

import torch

from . import _lib


class TerrainLayer:
    """Owns the device-side repack of one [K,G,G] nearest-triangle index and its mesh
    (reference assets: knn_terrain/ or knn_rocks/ {map_indices,triangles,vertices}.pt,
    camera.py:154-161, rock_detect.py:151-158)."""

    def __init__(self, map_indices_kgg, triangles, vertices, shift, res=0.1, device='cuda:0', sem=_lib.SEM_TORCH_CUDA,
                 index_only=False):
        """index_only: no block / superblock lists (RVB_LAYER_INDEX_ONLY) -- the layer of a Rock_Detection, whose kernel scans
        the K-lists themselves; half the memory and a third of the build time."""
        lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise RuntimeError("rover_b200: TerrainLayer needs a CUDA device (there is no CPU path)")
        idx = map_indices_kgg.to(self.device)
        if idx.dtype != torch.int32 or idx.dim() != 3:
            raise ValueError("map_indices must be int32 [K,G,G]")
        # the view the reference indexes: [G,G,K] (camera.py:157-158); strides passed through, no copy here
        view = idx.swapaxes(0, 1).swapaxes(1, 2)
        tri = triangles.to(self.device, torch.int32).contiguous()
        ver = vertices.to(self.device, torch.float16).contiguous()
        shift = torch.as_tensor(shift, dtype=torch.float32).flatten().cpu()
        self.res = float(res)
        self.shift = shift
        self.G0, self.G1, self.K = view.shape
        self.T, self.V = tri.shape[0], ver.shape[0]
        self.sem = sem
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(lib.rvb_terrain_create(C.byref(h), _lib.ptr(view), self.G0, self.G1, self.K,
                                              view.stride(0), view.stride(1), view.stride(2),
                                              _lib.ptr(tri), self.T, _lib.ptr(ver), self.V,
                                              self.res, float(shift[0]), float(shift[1]), sem,
                                              _lib.LAYER_INDEX_ONLY if index_only else 0, _lib.stream_of(idx)))
        self._h = h
        self._lib = lib

    @property
    def handle(self):
        if self._h is None:
            raise RuntimeError("TerrainLayer already destroyed")
        return self._h

    def bytes(self):
        return int(self._lib.rvb_terrain_bytes(self.handle))

    def release_index(self):
        """Frees the handle's K-contiguous index copy (more than half of the layer).  The production heightmap ray-cast does not
        read it; the per-pair cross-check variants, `cast_rays` and the rock kernel do and raise on this layer afterwards."""
        _lib.check(self._lib.rvb_terrain_release_index(self.handle))

    @property
    def has_index(self):
        return bool(self._lib.rvb_terrain_has_index(self.handle))

    @property
    def unbounded_triangles(self):
        """Triangles the shadow kernel has no culling bound for (rvb_terrain_unbounded_triangles)."""
        return int(self._lib.rvb_terrain_unbounded_triangles(self.handle))

    def close(self):
        if getattr(self, "_h", None) is not None:
            self._lib.rvb_terrain_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def build_knn_index(triangles, vertices, G, res, K, device='cuda:0'):
    """Device build of the [K,G,G] index (rover_utils.py:52-118 semantics, ties by triangle id)."""
    lib = _lib.load()
    dev = torch.device(device)
    tri = triangles.to(dev, torch.int32).contiguous()
    ver = vertices.to(dev, torch.float16).contiguous()
    coord = torch.arange(0, G * res, res, dtype=torch.float16)[:G].to(dev).contiguous()      # rover_utils.py:77-78
    if coord.shape[0] != G:
        raise ValueError("arange(0, G*res, res) produced fewer than G cell coordinates")
    out = torch.empty((K, G, G), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.rvb_build_knn_index(_lib.ptr(tri), tri.shape[0], _lib.ptr(ver), ver.shape[0], _lib.ptr(coord),
                                           _lib.ptr(coord), G, G, K, _lib.ptr(out), _lib.stream_of(out)))
    return out
