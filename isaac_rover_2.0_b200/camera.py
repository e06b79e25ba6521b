"""`Camera` -- mirror of tasks/utils/camera/camera.py:11-264: same constructor arguments, attributes and
`get_depths(positions, rotations) -> (distances f16 [N,P], pt f16 [N,P,3], sources f16 [N,P,3])`.
All arithmetic runs in rvb_heightmap_raycast (one fused launch)."""
import torch

from . import _lib
from .heightmap_distribution import Heightmap
from .terrain import TerrainLayer

ASSET_DIR = "tasks/utils/terrain/knn_terrain/"      # camera.py:156-160 (relative to CWD, like the reference)


class Camera():
    def __init__(self, device, shift, debug=False, assets=None, sem=_lib.SEM_TORCH_CUDA, variant=0, compact=False):
        """assets: optional (map_indices [K,G,G] int32, triangles [T,3] int32, vertices [V,3] fp16); when None
        the three .pt files are loaded from ASSET_DIR exactly as the reference does.
        compact: the layer gives back its K-contiguous copy of the index once its lists are built (TerrainLayer.release_index):
        5.0 GB instead of 8.2 GB on the benchmark world, same results; only the production variants (0, 3) run on such a layer."""
        self.debug = debug
        self.device = device
        self.partition = True
        self.heightmap = Heightmap(self.device)
        self.num_partitions = 4           # kept for interface parity; the kernel needs no VRAM partitioning
        self.horizontal = 0.1
        if assets is None:
            assets = tuple(torch.load(ASSET_DIR + f) for f in ("map_indices.pt", "triangles.pt", "vertices.pt"))
        mi, tri, ver = assets
        self.layer = TerrainLayer(mi, tri, ver, shift, res=self.horizontal, device=device, sem=sem)
        if compact:
            self.layer.release_index()
        self.map_indices = mi.to(device).swapaxes(0, 1).swapaxes(1, 2)
        self.triangles = tri.to(device)
        self.vertices = ver.to(device)
        self.heightmap_distribution = self.heightmap.get_distribution()
        self.num_exteroceptive = self.heightmap_distribution.shape[0]
        self.shift = shift
        self.dtype = torch.float16
        self.variant = variant
        self._col_a, self._col_b = self.heightmap.obs_columns(4)
        self.last_hit_slot = None
        self.timing = None          # set to a list to collect (start, end) CUDA events of every ray-cast launch
        self.last_hit_tri = None

    def get_num_exteroceptive(self):
        return self.num_exteroceptive

    def get_depths(self, positions, rotations, trig=None, want_hits=False, obs=None, want_pt=True):
        """trig (optional f32 [N,6]) overrides the device sin/cos of the negated euler angles (test hook);
        obs (optional f32 [N,>=4+ns+nd]) receives the fused sparse/dense columns (rover.py:324-325)."""
        _lib.require_cuda(positions, rotations)
        lib = _lib.load()
        pos = positions.to(torch.float32).contiguous()
        rot = rotations.to(torch.float32).contiguous()
        N, P = pos.shape[0], self.num_exteroceptive
        dev = pos.device
        dist = torch.empty((N, P), dtype=torch.float16, device=dev)
        pt = torch.empty((N, P, 3), dtype=torch.float16, device=dev) if want_pt else None
        src = torch.empty((N, P, 3), dtype=torch.float16, device=dev) if want_pt else None
        slot = torch.empty((N, P), dtype=torch.int32, device=dev) if want_hits else None
        tri = torch.empty((N, P), dtype=torch.int32, device=dev) if want_hits else None
        if trig is not None:
            trig = trig.to(torch.float32).contiguous()
        ev = None
        if self.timing is not None:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record(torch.cuda.current_stream(dev))
        with torch.cuda.device(dev):
            _lib.check(lib.rvb_heightmap_raycast(
                self.layer.handle, _lib.ptr(pos), _lib.ptr(rot), _lib.ptr(trig), _lib.ptr(self.heightmap_distribution), P, N,
                _lib.ptr(dist), _lib.ptr(slot), _lib.ptr(tri), _lib.ptr(pt), _lib.ptr(src),
                _lib.ptr(obs), 0 if obs is None else obs.stride(0), None, 0, 0, _lib.ptr(self._col_a if obs is not None else None),
                _lib.ptr(self._col_b if obs is not None else None), self.variant, _lib.stream_of(pos)))
        # variant 0 launches four kernels (classify, tiled kernel on the steep list, shadow, tiled kernel on the hand-back list),
        # variant 1 two (set-up + cast), variants 2/3 one
        if self.variant != 0:
            _lib.launch_count -= 2 if self.variant == 1 else 3
        if ev is not None:
            ev[1].record(torch.cuda.current_stream(dev))
            self.timing.append(ev)
        self.last_hit_slot, self.last_hit_tri = slot, tri
        return dist, pt, src

    def cast_rays(self, sources, directions, want_hits=False):
        """Cast arbitrary fp16 rays [R,3] against this layer (the lookup + ray_distance + min of get_depths)."""
        return cast_rays(self.layer, sources, directions, want_hits)


def cast_rays(layer, sources, directions, want_hits=False):
    _lib.require_cuda(sources, directions)
    lib = _lib.load()
    s = sources.to(torch.float16).contiguous().reshape(-1, 3)
    d = directions.to(torch.float16).contiguous().reshape(-1, 3)
    R = s.shape[0]
    dist = torch.empty((R,), dtype=torch.float16, device=s.device)
    pt = torch.empty((R, 3), dtype=torch.float16, device=s.device)
    slot = torch.empty((R,), dtype=torch.int32, device=s.device) if want_hits else None
    tri = torch.empty((R,), dtype=torch.int32, device=s.device) if want_hits else None
    with torch.cuda.device(s.device):
        _lib.check(lib.rvb_cast_rays(layer.handle, _lib.ptr(s), _lib.ptr(d), R, _lib.ptr(dist), _lib.ptr(slot), _lib.ptr(tri),
                                     _lib.ptr(pt), _lib.stream_of(s)))
    return (dist, pt, slot, tri) if want_hits else (dist, pt)
