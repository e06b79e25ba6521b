"""The env order the heightmap ray-cast and the rock kernel cast envs in (build_env_order: tilted envs first, then by map position)
changes which CTA or warp computes an env, never what it computes: the fused step, the standalone ray-cast and the standalone rock
collision give, for an env set permuted by a fixed permutation, the same permutation of their outputs, bit for bit.  The sets
cover every key equal (all envs in one cell), the map's border and corner cells, steep / tilted / flat envs mixed, and sizes
below and above the one from which the last envs of the order are split over two CTAs (1184)."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import isaac_rover_b200
    return isaac_rover_b200


@pytest.fixture(scope="module")
def world(R):
    w = R.synth.make_world(length=20.0, nv=200, K=64, n_stones=8, seed=5, build_index=None)
    w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device="cuda:0").cpu()
    kr = min(w.K, w.rock_triangles.shape[0])
    w.rock_indices = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, kr, device="cuda:0").cpu()
    return w


def _state(R, world, N, placement):
    """make_env_state with envs rolled / pitched into three classes (steep: rays nearly horizontal, tilted, flat) and placed
    uniformly, all in one cell, or on the map's border and corner cells (and just beyond them)."""
    st = R.synth.make_env_state(world, N, seed=31 + N, margin=3.0)
    g = torch.Generator().manual_seed(N)
    k = torch.arange(N) % 3
    tilt = torch.where(k == 0, torch.full((N,), 1.25), torch.where(k == 1, torch.full((N,), 0.45), torch.full((N,), 0.05)))
    roll = tilt * torch.where(torch.rand(N, generator=g) < 0.5, -1.0, 1.0)
    pitch = (torch.rand(N, generator=g) - 0.5) * 0.1
    yaw = (torch.rand(N, generator=g) - 0.5) * 2 * math.pi
    st["quat"] = R.synth.euler_to_quat_wxyz(roll, pitch, yaw).float().contiguous()
    L = world.length
    if placement == "one_cell":
        st["pos"][:, 0] = 0.5 * L + 0.013
        st["pos"][:, 1] = 0.5 * L - 0.021
    elif placement == "edges":
        spots = torch.tensor([[0.0, 0.0], [L, L], [0.0, L], [L, 0.0], [0.01, 0.5 * L], [L - 0.01, 0.5 * L], [0.5 * L, 0.01],
                              [0.5 * L, L - 0.01], [-0.4, -0.4], [L + 0.4, L + 0.4], [-0.4, 0.5 * L], [0.5 * L, L + 0.4]])
        st["pos"][:, :2] = spots[torch.arange(N) % spots.shape[0]]
    return st


def _permuted(st, perm):
    return {k: v[perm].contiguous() for k, v in st.items()}


def _perm(N):
    return torch.randperm(N, generator=torch.Generator().manual_seed(1000 + N))


def _fused(R, world, st):
    task = R.synth.make_task(world, st, device="cuda:0", level=2)
    obs, rew, reset, extras = task.hot_step(st["actions"].cuda())
    torch.cuda.synchronize()
    N = st["pos"].shape[0]
    out = dict(obs=obs, rew=rew, reset=reset, collision=task.rock_collison, dist=task._fused["dist"], wheel=task._fused["wheel"],
               body=task._fused["body"])
    out.update({"extras." + k: v for k, v in extras.items() if torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == N})
    return {k: v.clone() for k, v in out.items()}


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.float16 else t.view(torch.int32) if t.dtype == torch.float32 else t


def _same_under(a, b, perm):
    """b (outputs of the permuted env set) == a[perm] bit for bit, per output"""
    p = perm.cuda()
    bad = [k for k in a if not torch.equal(_bits(b[k]), _bits(a[k][p]))]
    assert not bad, bad


@pytest.mark.parametrize("N", [1, 7, 300, 5000])
@pytest.mark.parametrize("placement", ["uniform", "one_cell", "edges"])
def test_fused_step_is_permutation_invariant(R, world, N, placement):
    st = _state(R, world, N, placement)
    perm = _perm(N)
    a = _fused(R, world, st)
    assert len([k for k in a if k.startswith("extras.")]) >= 6
    b = _fused(R, world, _permuted(st, perm))
    _same_under(a, b, perm)


@pytest.mark.parametrize("N", [1, 7, 300, 5000])
@pytest.mark.parametrize("placement", ["uniform", "one_cell", "edges"])
def test_standalone_raycast_and_rock_collision_are_permutation_invariant(R, world, N, placement):
    cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(world.map_indices, world.triangles, world.vertices))
    rock = R.Rock_Detection("cuda:0", torch.tensor([0, 0, 0.0]), assets=(world.rock_indices, world.rock_triangles, world.rock_vertices))
    width = int(max(cam._col_a.max(), cam._col_b.max())) + 1
    st = _state(R, world, N, placement)
    perm = _perm(N)

    def run(s):
        pos, joints = s["pos"].cuda(), s["joints"].cuda()
        eul = R.tensor_quat_to_eul(s["quat"].cuda())
        obs = torch.full((N, width), -3.0, device="cuda:0")
        cam.variant = 0
        d, _, _ = cam.get_depths(pos, eul, obs=obs, want_pt=False)
        wheel, body = rock.get_collisions(pos, eul, joints, want_collision=True)
        torch.cuda.synchronize()
        return {k: v.clone() for k, v in dict(dist=d, obs=obs, wheel=wheel, body=body, collision=rock.last_collision).items()}

    a = run(st)
    b = run(_permuted(st, perm))
    _same_under(a, b, perm)
    if placement == "uniform" and N >= 300:
        cam.variant = 3                                       # the tiled kernel, which casts in index order: the same results
        pos = st["pos"].cuda()
        obs = torch.full((N, width), -3.0, device="cuda:0")
        d, _, _ = cam.get_depths(pos, R.tensor_quat_to_eul(st["quat"].cuda()), obs=obs, want_pt=False)
        torch.cuda.synchronize()
        assert torch.equal(d.view(torch.int16), a["dist"].view(torch.int16)) and torch.equal(obs.view(torch.int32), a["obs"].view(torch.int32))
        cam.variant = 0
