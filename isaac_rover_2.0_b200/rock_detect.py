"""`Rock_Detection` -- mirror of tasks/utils/rock_detection/rock_detect.py:9-401:
`get_collisions(positions, rotations, joint_states) -> (wheel_dist f16 [N,24], body_dist f16 [N,2])`."""
import torch

from . import _lib
from .terrain import TerrainLayer

ASSET_DIR = "tasks/utils/terrain/knn_rocks/"        # rock_detect.py:153-157


class Rock_Detection():
    def __init__(self, device, shift, debug=False, assets=None, sem=_lib.SEM_TORCH_CUDA):
        self.debug = debug
        self.device = device
        self.partition = True
        self.num_partitions = 1
        self.horizontal = 0.1
        if assets is None:
            assets = tuple(torch.load(ASSET_DIR + f) for f in ("map_indices.pt", "triangles.pt", "vertices.pt"))
        mi, tri, ver = assets
        # the rock kernel scans the K-lists themselves: no block / superblock lists for this layer
        self.layer = TerrainLayer(mi, tri, ver, shift, res=self.horizontal, device=device, sem=sem, index_only=True)
        self.rock_indices = mi.to(device).swapaxes(0, 1).swapaxes(1, 2)
        self.triangles = tri.to(device)
        self.vertices = ver.to(device)
        self.shift = shift
        self.dtype = torch.float16
        self.last_hit_tri = None
        self.last_collision = None
        self.last_rays = None

    def get_collisions(self, positions, rotations, joint_states, trig=None, want_hits=False, want_collision=False,
                       want_rays=False, joint_trig=None):
        _lib.require_cuda(positions, rotations, joint_states)
        lib = _lib.load()
        pos = positions.to(torch.float32).contiguous()
        rot = rotations.to(torch.float32).contiguous()
        jnt = joint_states.to(torch.float32).contiguous()
        if jnt.dim() != 2 or jnt.shape[1] != 13:
            raise ValueError("joint_states must be [N,13] (rock_detect.py:174-188)")
        N, dev = pos.shape[0], pos.device
        wheel = torch.empty((N, 24), dtype=torch.float16, device=dev)
        body = torch.empty((N, 2), dtype=torch.float16, device=dev)
        tri = torch.empty((N, 26), dtype=torch.int32, device=dev) if want_hits else None
        col = torch.empty((N,), dtype=torch.int64, device=dev) if want_collision else None
        rays = torch.empty((N, 26, 6), dtype=torch.float16, device=dev) if want_rays else None
        if trig is not None:
            trig = trig.to(torch.float32).contiguous()
        if joint_trig is not None:          # f32 [N,18]: sin, cos of joints 0..8 (tests: the oracle's values, for bit-identical rays)
            joint_trig = joint_trig.to(torch.float32).contiguous()
            if tuple(joint_trig.shape) != (N, 18):
                raise ValueError("joint_trig must be [N,18]")
        with torch.cuda.device(dev):
            _lib.check(lib.rvb_rock_collision(self.layer.handle, _lib.ptr(pos), _lib.ptr(rot), _lib.ptr(trig), _lib.ptr(jnt),
                                              _lib.ptr(joint_trig), N, _lib.ptr(wheel), _lib.ptr(body), _lib.ptr(tri), _lib.ptr(col),
                                              _lib.ptr(rays), _lib.stream_of(pos)))
        self.last_hit_tri, self.last_collision, self.last_rays = tri, col, rays
        return wheel, body
