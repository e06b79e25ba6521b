"""The tuning knobs of the heightmap ray-cast (DESIGN.md 6, "Tuning knobs") on the GPU: every knob at in-range values gives the
default's results bit for bit, a bad value fails the call before anything is launched, and the variables of the A/B switches
that were removed change nothing."""
import pytest
import torch

pytestmark = pytest.mark.gpu

KNOBS = ("RVB_SHADOW_TASK_RAYS", "RVB_SHADOW_SH", "RVB_SHADOW_SPLIT", "RVB_COS_STEEP", "RVB_SHADOW_FORCE", "RVB_SHADOW_DBG")
REMOVED = {"RVB_SHADOW_SPEC": "3", "RVB_SHADOW_BULK": "1746", "RVB_SHADOW_BIG": "1", "RVB_SHADOW_PAD": "40000",
           "RVB_ROCK_CTAS": "1", "RVB_TC_TAIL": "0", "RVB_POLICY_PDL": "0"}


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import isaac_rover_b200
    return isaac_rover_b200


@pytest.fixture(scope="module")
def world(R):
    w = R.synth.make_world(length=20.0, nv=200, K=64, n_stones=8, seed=5, build_index=None)
    w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device="cuda:0")
    kr = min(w.K, w.rock_triangles.shape[0])
    w.rock_indices = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, kr, device="cuda:0").cpu()
    w.map_indices = w.map_indices.cpu()
    return w


@pytest.fixture(scope="module")
def scene(R, world):
    """Camera + 1536 envs (more than the 1184 from which the tail split is on by default), a third of them strongly tilted so
    that the steep list and the hand-back list are used."""
    cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(world.map_indices, world.triangles, world.vertices))
    st = R.synth.make_env_state(world, 1536, seed=12, margin=3.0)
    eul = R.tensor_quat_to_eul(st["quat"].cuda())
    g = torch.Generator().manual_seed(7)
    eul[:512, :2] += ((torch.rand(512, 2, generator=g) - 0.5) * 2.4).cuda()
    width = int(max(cam._col_a.max(), cam._col_b.max())) + 1
    return cam, st["pos"].cuda(), eul, width


def _cast(scene, fill=0.0):
    cam, pos, eul, width = scene
    obs = torch.full((pos.shape[0], width), fill, device="cuda:0")
    cam.variant = 0
    d, _, _ = cam.get_depths(pos, eul, obs=obs, want_pt=False)
    torch.cuda.synchronize()
    return d.view(torch.int16).clone(), obs


@pytest.mark.parametrize("name,values", [("RVB_SHADOW_TASK_RAYS", ("1", "32")), ("RVB_SHADOW_SH", ("0", "3")),
                                         ("RVB_SHADOW_SPLIT", ("0", "100000")), ("RVB_COS_STEEP", ("0", "1")),
                                         ("RVB_SHADOW_FORCE", ("0", "1")), ("RVB_SHADOW_DBG", ("0", "1"))])
def test_knobs_in_range_change_no_result(R, scene, monkeypatch, name, values):
    assert name in KNOBS
    for k in KNOBS + tuple(REMOVED):
        monkeypatch.delenv(k, raising=False)
    d0, obs0 = _cast(scene)
    assert (d0 != 0x4980).float().mean() > 0.3                     # the envs see terrain: hits, not only misses
    for v in values:
        monkeypatch.setenv(name, v)
        d, obs = _cast(scene)
        assert torch.equal(d, d0), (name, v)
        assert torch.equal(obs.view(torch.int32), obs0.view(torch.int32)), (name, v)


@pytest.mark.parametrize("name,bad", [("RVB_SHADOW_SH", "4"), ("RVB_SHADOW_SH", "-1"), ("RVB_SHADOW_SH", "x"),
                                      ("RVB_SHADOW_TASK_RAYS", "0"), ("RVB_SHADOW_TASK_RAYS", "33"), ("RVB_SHADOW_TASK_RAYS", "12abc"),
                                      ("RVB_SHADOW_SPLIT", "-1"), ("RVB_SHADOW_SPLIT", "1.5"), ("RVB_SHADOW_SPLIT", ""),
                                      ("RVB_COS_STEEP", "1.5"), ("RVB_COS_STEEP", "-0.1"), ("RVB_COS_STEEP", "nan"),
                                      ("RVB_COS_STEEP", "0.7x"), ("RVB_SHADOW_FORCE", "2"), ("RVB_SHADOW_FORCE", "yes"),
                                      ("RVB_SHADOW_DBG", "2"), ("RVB_SHADOW_DBG", " 1")])
def test_bad_knob_values_fail_before_any_launch(R, scene, monkeypatch, name, bad):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv(name, bad)
    cam, pos, eul, width = scene
    obs = torch.full((pos.shape[0], width), -7.0, device="cuda:0")
    for variant in (0, 3):
        cam.variant = variant
        with pytest.raises(RuntimeError, match=name):
            cam.get_depths(pos, eul, obs=obs, want_pt=False)
    torch.cuda.synchronize()
    assert bool((obs == -7.0).all())                               # nothing was launched
    monkeypatch.delenv(name)
    _cast(scene)                                                     # the library is still usable


def _step_and_policy(R, world):
    st = R.synth.make_env_state(world, 1024, seed=21, margin=3.0)
    task = R.synth.make_task(world, st, device="cuda:0", level=2)
    obs, rew, reset, _ = task.hot_step(st["actions"].cuda())
    torch.manual_seed(1)
    net = R.model.NetworkInfo([256, 160, 128], [80, 60], [80, 60], [80, 60], "leakyrelu")
    info = R.model.ObserverationInfo(4, 634, 1112, 0)
    actor = R.model.StochasticActorHeightmap(1750, 2, net, info, device="cuda:0")
    critic = R.model.DeterministicHeightmap(1750, 2, net, info, device="cuda:0")
    mean, value = R.model.compute_pair(actor, critic, obs)
    torch.cuda.synchronize()
    out = dict(obs=obs, rew=rew, reset=reset, collision=task.rock_collison, wheel=task._fused["wheel"], body=task._fused["body"],
               mean=mean, value=value)
    return {k: v.clone() for k, v in out.items()}


def test_removed_switches_change_nothing(R, world, monkeypatch):
    """The variables of the A/B switches the library no longer has, each set to a value that used to re-route a kernel: the env
    step (ray-cast + rock kernel) and the policy / value pair stay bit-identical."""
    for k in KNOBS + tuple(REMOVED):
        monkeypatch.delenv(k, raising=False)
    ref = _step_and_policy(R, world)
    for name, v in REMOVED.items():
        monkeypatch.setenv(name, v)
        got = _step_and_policy(R, world)
        for k in ref:
            assert torch.equal(got[k], ref[k]), (name, k)
        monkeypatch.delenv(name)
