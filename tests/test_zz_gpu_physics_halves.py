"""RoverTask.pre_physics_step_fused / post_physics_step_fused (rvb_env_pre / rvb_env_post): the fused step split at the simulator's
boundary, for the loop obs_t -> policy -> pre_physics_step(a_t) -> physics -> post_physics_step() -> obs_{t+1}.  Both sides of every
comparison run the same device code, so every comparison is torch.equal."""
import pytest
import torch

pytestmark = pytest.mark.gpu

N = 300


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import isaac_rover_b200
    return isaac_rover_b200


@pytest.fixture(scope="module")
def world20(R):
    return R.synth.make_world(length=20.0, nv=72, K=200, n_stones=12, seed=1)


def _resetting(R, task):
    """Give the task's view the simulator's pose reset: envs in the mask go back to initial_pos with a quaternion of their own,
    different from the one they had, so that a post half which took rover_rot after the reset would see another pose."""
    base = R.synth.SyntheticRoverView

    class ResettingView(base):
        reset_quat = R.synth.euler_to_quat_wxyz(torch.tensor([0.3]), torch.tensor([-0.2]), torch.tensor([1.0])).float().cuda()

        def reset_idx_masked(self, mask, initial_pos):
            m = (mask != 0).unsqueeze(1)
            self.pos = torch.where(m, initial_pos, self.pos).contiguous()
            self.quat = torch.where(m, self.reset_quat.expand_as(self.quat), self.quat).contiguous()

    task._rover.__class__ = ResettingView
    return task


def _physics(views, k):
    """Stand-in for the simulator's step: the same pose and joint change, applied to every view."""
    g = torch.Generator().manual_seed(500 + k)
    n = views[0].pos.shape[0]
    dpos = ((torch.rand(n, 3, generator=g) - 0.5) * 0.2).cuda()
    dq = ((torch.rand(n, 4, generator=g) - 0.5) * 0.3).cuda()
    dj = ((torch.rand(n, 13, generator=g) - 0.5) * 0.1).cuda()
    for v in views:
        v.pos = (v.pos + dpos).contiguous()
        q = v.quat + dq
        v.quat = (q / q.norm(dim=1, keepdim=True)).contiguous()
        v.joints = (v.joints + dj).contiguous()


def _state(t, level):
    out = dict(obs=t.obs_buf, rew=t.rew_buf, reset=t.reset_buf, progress=t.progress_buf, stats=t.stats, rock=t.rock_collison,
               lin=t.linear_velocity.tracker, ang=t.angular_velocity.tracker, pos_t=t.joint_position_targets,
               vel_t=t.joint_velocity_targets, view_pos_t=t._rover.position_targets, view_vel_t=t._rover.velocity_targets,
               heading=t.heading_diff, target=t.target_positions, counters=t.reset_counters, rover_rot=t.rover_rot,
               rover_rotation=t.rover_rotation)
    if level >= 2:
        out.update(wheel=t.rock_wheel_dist, body=t.rock_body_dist)
    out.update({"extras." + k: v for k, v in t.extras.items()})
    return {k: v.clone() for k, v in out.items()}


def _same(a, b):
    assert a.keys() == b.keys()
    bad = [k for k in a if not torch.equal(a[k], b[k])]
    assert not bad, bad


@pytest.mark.parametrize("level", [1, 2])
def test_fused_halves_equal_reference_loop(R, world20, level):
    """Four steps of actions -> pre half -> physics -> post half: the fused pair gives what pre_physics_step_device +
    post_physics_step give, with pose resets by the view and envs resetting during the run."""
    st = R.synth.make_env_state(world20, N, seed=41)
    tasks = [_resetting(R, R.synth.make_task(world20, st, device="cuda:0", level=level)) for _ in range(2)]
    for t in tasks:
        t.reset_buf.zero_()
        t.reset_buf[::7] = 1
    g = torch.Generator().manual_seed(3)
    resets_seen = 0
    for k in range(4):
        act = (torch.rand(N, 2, generator=g) * 2 - 1).cuda()
        fused, ref = tasks
        resets_seen += int(ref.reset_buf.sum()) if k > 0 else 0
        fused.pre_physics_step_fused(act)
        ref.pre_physics_step_device(act)
        _physics([fused._rover, ref._rover], k)
        fused.post_physics_step_fused()
        ref.post_physics_step()
        torch.cuda.synchronize()
        _same(_state(fused, level), _state(ref, level))
    assert 0 < resets_seen < 3 * N                     # envs reset during the run (the view then writes another quaternion)


def test_rover_rot_is_the_pre_physics_pose(R, world20):
    """is_done reads the pose of the pre half: an env that was tilted past the limit before physics and is level after it is
    reset, an env the other way round is not."""
    n = 64
    st = R.synth.make_env_state(world20, n, seed=43)
    task = R.synth.make_task(world20, st, device="cuda:0", level=1)
    task.reset_buf.zero_()
    task.progress_buf.fill_(10)
    task.target_positions = task._rover.pos.clone()
    task.target_positions[:, 0] += 3.0
    yaw = torch.zeros(n)
    tilted = R.synth.euler_to_quat_wxyz(torch.full((n,), 1.2), torch.zeros(n), yaw).float().cuda()
    level = R.synth.euler_to_quat_wxyz(torch.zeros(n), torch.zeros(n), yaw).float().cuda()
    even = (torch.arange(n) % 2 == 0).cuda().unsqueeze(1)
    task._rover.quat = torch.where(even, tilted, level).contiguous()
    task.pre_physics_step_fused(torch.zeros(n, 2, device="cuda:0"))
    task._rover.quat = torch.where(even, level, tilted).contiguous()
    task.post_physics_step_fused()
    reset = task.reset_buf.cpu()
    assert torch.equal(reset[0::2], torch.ones(n // 2, dtype=torch.long))
    assert torch.equal(reset[1::2], torch.zeros(n // 2, dtype=torch.long))
    assert torch.all(task.rover_rotation[:, 0].abs()[1::2] > 1.1)             # the observation did see the tilted post pose


def test_packed_post_half(R, world20):
    """obs16_buf on the post half: the fp16 heightmap columns widened equal the f32 run's obs_buf[:, 4:]; the proprioceptive
    columns, rew and reset are unchanged.  Observation hooks together with obs16_buf are refused."""
    st = R.synth.make_env_state(world20, N, seed=45)
    t32, t16 = [_resetting(R, R.synth.make_task(world20, st, device="cuda:0", level=2)) for _ in range(2)]
    t16.obs16_buf = torch.zeros((N, t16.num_observations - 4), dtype=torch.float16, device="cuda:0")
    g = torch.Generator().manual_seed(4)
    for k in range(3):
        act = (torch.rand(N, 2, generator=g) * 2 - 1).cuda()
        for t in (t32, t16):
            t.pre_physics_step_fused(act)
        _physics([t32._rover, t16._rover], k)
        obs, rew, reset, _ = t32.post_physics_step_fused()
        _, rew2, reset2, _ = t16.post_physics_step_fused()
        torch.cuda.synchronize()
        assert torch.equal(t16.obs16_buf.float(), obs[:, 4:]) and torch.equal(t16.obs_buf[:, :4], obs[:, :4])
        assert torch.equal(rew, rew2) and torch.equal(reset, reset2)
    t16.obs_hooks = R.hooks.ObsHooks(t16.num_observations, device="cuda:0")
    with pytest.raises(RuntimeError, match="observation hooks work on obs_buf"):
        t16.post_physics_step_fused()


@pytest.mark.parametrize("level", [1, 2])
def test_unchanged_pose_equals_hot_step(R, world20, level):
    """With no physics between the halves, the pair in a simulator loop's order (action half, then reset half) gives the bits of
    hot_step(device_reset=True), which runs the reset half first and then the action half (this view moves no env on a reset, so
    both orders read the same pose)."""
    st = R.synth.make_env_state(world20, N, seed=47)
    pair, step = [R.synth.make_task(world20, st, device="cuda:0", level=level) for _ in range(2)]
    g = torch.Generator().manual_seed(5)
    for k in range(3):
        act = (torch.rand(N, 2, generator=g) * 2 - 1).cuda()
        pair.pre_physics_step_fused(act)
        pair.post_physics_step_fused()
        step.hot_step(act, device_reset=True)
        torch.cuda.synchronize()
        _same(_state(pair, level), _state(step, level))


def test_not_playing_only_counts_progress(R, world20):
    """rl_task.py:241 increments progress before the is_playing guard (:250); nothing else of the post half runs."""
    st = R.synth.make_env_state(world20, N, seed=49)
    task = R.synth.make_task(world20, st, device="cuda:0", level=2)
    task.pre_physics_step_fused(torch.zeros(N, 2, device="cuda:0"))
    task.post_physics_step_fused()
    torch.cuda.synchronize()

    class World:
        playing = False

        def is_playing(self):
            return self.playing

    class Env:
        _world = World()

    task._env = Env()
    before = _state(task, 2)
    task.post_physics_step_fused()
    torch.cuda.synchronize()
    after = _state(task, 2)
    assert torch.equal(after.pop("progress"), before.pop("progress") + 1)
    _same(after, before)
