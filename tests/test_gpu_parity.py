"""GPU parity tests (run on the B200 box): CUDA kernels behind the C ABI vs (a) the golden vectors the
reference itself produced, (b) the oracle restatement on the CPU and on the GPU.

Tolerances (BASELINE.json north_star): bit-exact for fp16 distances given identical trig inputs, hit
slots / triangle ids, collision flags, reset masks, validity flags; <= 1e-5 relative for fp32 heights,
kinematics and rewards (libm atan2/asin/sin/cos differ by an ulp between torch-CPU, torch-CUDA and here).
"""
import math
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
RTOL = 1e-5
ATOL = 1e-6


def _skip_without_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.fixture(scope="module")
def R():
    _skip_without_gpu()
    import isaac_rover_b200
    return isaac_rover_b200


@pytest.fixture(scope="module")
def O():
    import rover_oracle
    return rover_oracle


@pytest.fixture(scope="module")
def golden():
    return torch.load(os.path.join(HERE, "golden", "rover_golden.pt"))


@pytest.fixture(scope="module")
def gcam(R, golden):
    w = golden["world"]
    return R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(w["map_indices"].to(torch.int32), w["triangles"], w["vertices"]),
                    sem=R.SEM_TORCH_CPU)


@pytest.fixture(scope="module")
def grock(R, golden):
    w = golden["world"]
    return R.Rock_Detection("cuda:0", torch.tensor([0, 0, 0.0]),
                            assets=(w["rock_indices"].to(torch.int32), w["rock_triangles"], w["rock_vertices"]), sem=R.SEM_TORCH_CPU)


def joint_trig(joints):
    """f32 [N,18]: sin, cos of joints 0..8, computed by torch on the device the tensor lives on (CPU for the golden vectors)."""
    j = joints[:, :9].float()
    return torch.stack((torch.sin(j), torch.cos(j)), 2).reshape(j.shape[0], 18)


def bits(t):
    return t.view(torch.int16) if t.dtype == torch.float16 else t


def assert_bits_equal(a, b, what):
    a, b = a.cpu(), b.cpu()
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, tuple(a.shape), tuple(b.shape))
    neq = bits(a) != bits(b)
    if a.dtype.is_floating_point:                      # -0 == +0 and NaN == NaN are still bit comparisons here
        pass
    assert not neq.any(), "%s: %d of %d elements differ, first at %s: %s vs %s" % (
        what, int(neq.sum()), neq.numel(), neq.nonzero()[0].tolist(), a[neq][0].item(), b[neq][0].item())


def close(a, b, what, rtol=RTOL, atol=ATOL):
    a, b = a.cpu().double(), b.cpu().double()
    err = (a - b).abs()
    tol = atol + rtol * b.abs()
    bad = err > tol
    bad &= ~(a.isnan() & b.isnan())
    bad &= ~((a == b))                                 # equal infinities
    assert not bad.any(), "%s: %d of %d beyond tolerance, worst abs err %g" % (what, int(bad.sum()), bad.numel(), err[bad].max())


# --------------------------------------------------------------------------- golden vectors (reference outputs)
def test_golden_pattern(R, golden):
    hm = R.Heightmap("cuda:0")
    assert torch.equal(hm.get_distribution().cpu(), golden["ref_pattern"])
    assert torch.equal(hm.coarse_idx.cpu(), golden["ref_coarse_idx"])
    assert torch.equal(hm.fine_idx.cpu(), golden["ref_fine_idx"])
    assert (hm.get_num_sparse_vector(), hm.get_num_dense_vector()) == (634, 1112)      # teacher_loader.py:47-48


@pytest.mark.parametrize("variant", [0, 1, 2, 3])
def test_golden_get_depths(R, golden, gcam, variant):
    gcam.variant = variant
    dist, pt, src = gcam.get_depths(golden["in_pos"].cuda(), golden["ref_euler"].cuda(), trig=golden["trig"].cuda(), want_hits=True)
    assert_bits_equal(src, golden["ref_sources"], "sources")
    assert_bits_equal(dist, golden["ref_dist"], "distances")
    assert_bits_equal(pt, golden["ref_pt"], "intersection points")
    assert_bits_equal(gcam.last_hit_slot, golden["oracle_slot"], "hit slot")
    assert_bits_equal(gcam.last_hit_tri, golden["oracle_tri"], "hit triangle")
    gcam.variant = 0


def test_golden_rock_detection(R, golden, grock):
    """With the reference's trigonometry injected (body and joints) everything is bit-identical: rays, distances, collision flags.
    With the device's own sinf / cosf of the joint angles the rays stay within one fp16 ulp."""
    wheel, body = grock.get_collisions(golden["in_pos"].cuda(), golden["ref_euler"].cuda(), golden["in_joints"].cuda(),
                                       trig=golden["trig"].cuda(), joint_trig=joint_trig(golden["in_joints"]).cuda(),
                                       want_collision=True, want_rays=True)
    rays = grock.last_rays.cpu()
    assert_bits_equal(rays[:, :, 0:3], golden["ref_rock_sources"], "rock ray sources")
    assert_bits_equal(rays[:, :, 3:6], golden["ref_rock_dirs"], "rock ray directions")
    assert_bits_equal(wheel, golden["ref_wheel"], "wheel distances")
    assert_bits_equal(body, golden["ref_body"], "body distances")
    assert torch.equal(grock.last_collision.cpu(), golden["ref_rock_collision"])
    # device libm for the joint angles
    grock.get_collisions(golden["in_pos"].cuda(), golden["ref_euler"].cuda(), golden["in_joints"].cuda(), trig=golden["trig"].cuda(),
                         want_rays=True)
    rays = grock.last_rays.cpu()
    ds = (rays[:, :, 0:3].float() - golden["ref_rock_sources"].float()).abs().max().item()
    dd = (rays[:, :, 3:6].float() - golden["ref_rock_dirs"].float()).abs().max().item()
    assert ds <= 2e-3 and dd <= 1e-3, (ds, dd)


def test_golden_rock_cast_given_reference_rays(R, golden, grock):
    s, d = golden["ref_rock_sources"].cuda(), golden["ref_rock_dirs"].cuda()
    dist, pt = R.cast_rays(grock.layer, s, d)
    refw = torch.cat((golden["ref_wheel"], golden["ref_body"]), 1)
    assert_bits_equal(dist.reshape(refw.shape), refw, "rock distances from reference rays")
    task_col = torch.empty(refw.shape[0], dtype=torch.long, device="cuda")
    lib = R._lib.load()
    w, b = dist.reshape(refw.shape)[:, :24].contiguous(), dist.reshape(refw.shape)[:, 24:].contiguous()
    R._lib.check(lib.rvb_check_collision(R._lib.ptr(w), R._lib.ptr(b), w.shape[0], R._lib.ptr(task_col), None))
    torch.cuda.synchronize()
    assert torch.equal(task_col.cpu(), golden["ref_rock_collision"])


@pytest.mark.parametrize("K", [1, 2, 7, 37, 64, 65, 100, 129, 200])
def test_rock_kernel_candidate_counts(R, K):
    """The rock kernel (K / 64 full warp iterations per ray + the rays' tails scanned together, several rays per warp iteration)
    against the per-pair kernel behind cast_rays on the rays it generated itself: distances and hit triangles bit for bit for
    every split of K into full iterations and tail."""
    w = R.synth.make_world(length=12.0, nv=44, K=200, n_stones=8, seed=3, build_index=None)
    kr = min(K, w.rock_triangles.shape[0])
    idx = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, kr, device="cuda:0")
    rock = R.Rock_Detection("cuda:0", torch.tensor([0, 0, 0.0]), assets=(idx, w.rock_triangles, w.rock_vertices))
    st = {k: v.cuda() for k, v in R.synth.make_env_state(w, 300, seed=21 + K, margin=2.0).items()}
    g = torch.Generator().manual_seed(K)
    stones = w.stone_info[:, :2].float()
    st["pos"][:200, :2] = (stones[torch.randint(0, stones.shape[0], (200,), generator=g)] + torch.rand(200, 2, generator=g) - 0.5).cuda()
    eul = R.tensor_quat_to_eul(st["quat"])
    wheel, body = rock.get_collisions(st["pos"], eul, st["joints"], want_hits=True, want_rays=True)
    rays = rock.last_rays.reshape(-1, 6)
    dist, pt, slot, tri = R.cast_rays(rock.layer, rays[:, 0:3], rays[:, 3:6], want_hits=True)
    mine = torch.cat((wheel, body), 1).reshape(-1)
    assert torch.equal(bits(mine), bits(dist))
    assert torch.equal(rock.last_hit_tri.reshape(-1), tri)
    assert (mine != 11).float().mean() > 0.02 or K < 7


def test_golden_ray_distance(R, golden):
    k, pt = R.ray_distance(golden["in_rd_src"].cuda(), golden["in_rd_dir"].cuda(), golden["in_rd_tri"].cuda())
    assert_bits_equal(k, golden["ref_rd_k"], "known-answer k")
    assert_bits_equal(pt, golden["ref_rd_pt"], "known-answer pt")
    assert k[0].item() == 1.0 and k[1].item() == -1.0 and k[2].item() == 11.0 and k[3].item() == 11.0 and k[4].item() == 11.0
    k, pt = R.ray_distance(golden["in_rr_src"].cuda(), golden["in_rr_dir"].cuda(), golden["in_rr_tri"].cuda())
    assert_bits_equal(k, golden["ref_rr_k"], "random-pair k")
    assert_bits_equal(pt, golden["ref_rr_pt"], "random-pair pt")


def test_golden_quat_to_euler(R, golden):
    close(R.tensor_quat_to_eul(golden["in_quat"].cuda()), golden["ref_euler"], "euler")


def test_golden_ackermann(R, golden):
    for lin, ang, rs, rv in ((golden["in_ka_lin"], golden["in_ka_ang"], golden["ref_ka_steer"], golden["ref_ka_vel"]),
                             (golden["in_actions"][:, 0], golden["in_actions"][:, 1], golden["ref_steer"], golden["ref_vel"])):
        steer, vel = R.Ackermann(lin.cuda(), ang.cuda(), "cuda:0", sem=R.SEM_TORCH_CPU)
        close(steer, rs, "steering angles")
        close(vel, rv, "motor velocities")
    steer, vel = R.Ackermann(torch.tensor([0.5], device="cuda"), torch.tensor([0.2], device="cuda"))
    close(steer, torch.tensor([[0.20421, 0.15067, 0, 0, -0.19193, -0.14151]]), "SURVEY known answer steer", rtol=1e-4, atol=1e-5)
    close(vel, torch.tensor([[2.1599, 2.9181, 2.0530, 2.9470, 2.1546, 2.9141]]), "SURVEY known answer vel", rtol=1e-4)
    # strided column views of actions[N,2] (rover.py:391)
    a = golden["in_actions"].cuda()
    s2, v2, pt, vt = R.Ackermann(a[:, 0], a[:, 1], "cuda:0", sem=R.SEM_TORCH_CPU, want_targets=True)
    close(s2, golden["ref_steer"], "strided steer")
    assert torch.equal(pt, s2[:, [1, 5, 0, 4]]) and torch.equal(vt, v2[:, [1, 3, 5, 0, 2, 4]])


def _golden_task(R, golden, level):
    w = golden["world"]
    world = R.synth.World(length=w["length"], res=w["res"], G=w["G"], K=w["K"], vertices=w["vertices"], triangles=w["triangles"],
                          rock_vertices=w["rock_vertices"], rock_triangles=w["rock_triangles"], stone_info=w["stone_info6"],
                          heightmap=w["heightmap"], hm_res=w["hm_res"], map_indices=w["map_indices"].to(torch.int32),
                          rock_indices=w["rock_indices"].to(torch.int32))
    st = {k[3:]: v for k, v in golden.items() if k.startswith("in_") and k[3:] in
          ("pos", "quat", "joints", "actions", "prev_actions", "target", "progress")}
    task = R.synth.make_task(world, st, level=level, sem=R.SEM_TORCH_CPU)
    task.apply_actions(st["actions"].cuda())
    task.rover_rot = R.tensor_quat_to_eul(st["quat"].cuda())
    return task


def test_golden_task_step(R, golden):
    task = _golden_task(R, golden, 2)
    task.parity_trig = golden["trig"].cuda()                          # the reference run's sin / cos (torch-CPU libm)
    task.parity_joint_trig = joint_trig(golden["in_joints"]).cuda()
    obs = task.get_observations()["rover_view"]["obs_buf"]
    ref = golden["ref_obs"]
    close(obs[:, 0:4], ref[:, 0:4], "proprioceptive obs")
    close(task.heading_diff, golden["ref_heading"], "heading")
    assert torch.equal(obs[:, 4:].cpu(), ref[:, 4:]), "heightmap observation columns"
    assert torch.equal(task.rock_collison.cpu(), golden["ref_rock_collision"])
    task.calculate_metrics()
    task.is_done()
    close(task.rew_buf, golden["ref_rew"], "rew_buf")
    assert torch.equal(task.reset_buf.cpu(), golden["ref_reset"])
    for k, v in golden["ref_extras"].items():
        if v.dtype == torch.long:
            assert torch.equal(task.extras[k].cpu(), v), k
        else:
            close(task.extras[k], v, "extras." + k)
    st = task.stats.cpu()
    assert st[0].item() == 8 and st[8].item() == task.reset_buf.sum().item()
    assert abs(st[1].item() - task.rew_buf.double().sum().item()) < 1e-9
    task1 = _golden_task(R, golden, 1)
    task1.parity_trig = golden["trig"].cuda()
    task1.get_observations()
    task1.calculate_metrics()
    task1.is_done()
    close(task1.rew_buf, golden["ref_rew_level1"], "rew_buf level 1")
    assert torch.equal(task1.reset_buf.cpu(), golden["ref_reset_level1"])
    # the device's own libm instead of the injected trig: a measured property, not the gate -- the columns that differ are one
    # fp16 ulp of a source coordinate away
    task2 = _golden_task(R, golden, 2)
    obs2 = task2.get_observations()["rover_view"]["obs_buf"]
    hm_same = (obs2[:, 4:].cpu() == ref[:, 4:]).float().mean().item()
    assert hm_same >= 0.99, "heightmap obs columns equal fraction %g with device trig" % hm_same


def test_golden_stones_and_heights(R, golden):
    task = _golden_task(R, golden, 2)
    assert torch.equal(task.stone_info.cpu(), golden["ref_stone7"])
    near, flag, cnt = task.nearest_stone_edge(task.target_positions[:, 0:2], 1.0)
    close(near, golden["ref_goal_nearest"], "goal nearest stone edge", rtol=1e-5, atol=1e-5)
    ref_flag = (golden["ref_goal_nearest"] <= 1.0).long()
    unstable = (golden["ref_goal_nearest"] - 1.0).abs() < 1e-4
    assert torch.equal(flag.cpu()[~unstable], ref_flag[~unstable])
    near, _, _ = task.nearest_stone_edge(golden["in_spawn_pos"].cuda()[:, 0:2], 1.4)
    close(near, golden["ref_many_nearest"], "nearest stone edge (matmul formulation)", rtol=1e-5, atol=2e-5)
    # cdist's DIRECT path (<= 25 rows on both sides, what rover.py:655 runs for a small env count): bit-exact spawn positions
    sg = torch.load(os.path.join(HERE, "golden", "spawn_direct_golden.pt"))
    for case in sg["cases"]:
        task.stone_info = case["stone7"].cuda()
        moved = task.avoid_pos_rock_collision(case["in_pos"].cuda().clone())
        assert torch.equal(moved.cpu(), case["ref_pos"]), "spawn validation, direct cdist path"
        near, flag, _ = task.nearest_stone_edge(case["in_pos"].cuda()[:, 0:2], 1.0)
        # the golden distances come from torch-CPU, whose vectorised float32 sqrt is not correctly rounded (DESIGN.md section 2):
        # one ulp of slack on the distance, none on the validity flag (no golden distance sits within 1e-6 of the threshold)
        assert (case["ref_nearest"] - 1.0).abs().min().item() > 1e-6
        assert torch.allclose(near.cpu(), case["ref_nearest"], rtol=2.4e-7, atol=1e-7)
        assert torch.equal(flag.cpu(), (case["ref_nearest"] <= 1.0).long())
    task.stone_info = golden["ref_stone7"].cuda()
    # cdist's MATMUL path (> 25 rows; GEMM summation order unspecified, so a position can take one 0.05 m step more or less):
    # rows that differ must still satisfy the loop's invariants
    moved = task.avoid_pos_rock_collision(golden["in_spawn_pos"].cuda().clone()).cpu()
    ref = golden["ref_spawn_pos"]
    same = (moved == ref).all(1)
    assert torch.equal(moved[:, 1:], golden["in_spawn_pos"][:, 1:])                          # only x moves
    steps = (moved[:, 0] - golden["in_spawn_pos"][:, 0]).double() / 0.05
    assert (steps - steps.round()).abs().max().item() < 1e-3 and (steps >= -1e-3).all()      # by whole 0.05 m steps
    import rover_oracle as RO_
    final_near = RO_.nearest_stone_edge(moved[:, 0:2].double(), golden["ref_stone7"].double())
    assert (final_near > 1.4 - 1e-4).all()                                                    # every final position clears the stones
    assert ((moved[:, 0] - ref[:, 0]).abs() <= 0.05 + 1e-5).all()                             # at most one step from the reference's
    print("spawn validation (matmul path): %d / %d rows bit-equal to the reference" % (int(same.sum()), same.numel()))
    assert same.float().mean() >= 0.8
    h = task.get_pos_height(task.heightmap, ref[:, 0:2].cuda(), golden["world"]["hm_res"], 1, torch.tensor([0.0, 0.0]))
    assert_bits_equal(h, golden["ref_spawn_height"], "get_pos_height")


# --------------------------------------------------------------------------- oracle on CPU and on CUDA, larger world
@pytest.fixture(scope="module")
def world20(R):
    return R.synth.make_world(length=20.0, nv=72, K=200, n_stones=12, seed=1)


def _trig(euler):
    return torch.stack([f(-euler[:, a]) for a in range(3) for f in (torch.sin, torch.cos)], 1)


@pytest.mark.parametrize("N", [1, 6, 64])
def test_oracle_cpu_semantics_bit_exact(R, O, world20, N):
    w = world20
    st = R.synth.make_env_state(w, N, seed=100 + N)
    eul = O.quat_to_euler(st["quat"])
    pat, _, _ = O.heightmap_pattern()
    ref = O.get_depths(st["pos"], eul, pat, w.map_indices, w.triangles, w.vertices, torch.tensor([0, 0, 0.0]))
    cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(w.map_indices, w.triangles, w.vertices), sem=R.SEM_TORCH_CPU)
    for variant in (0, 1, 2, 3):
        cam.variant = variant
        dist, pt, src = cam.get_depths(st["pos"].cuda(), eul.cuda(), trig=_trig(eul).cuda(), want_hits=True)
        assert_bits_equal(src, ref["sources"], "sources v%d" % variant)
        assert_bits_equal(dist, ref["dist"], "dist v%d" % variant)
        assert_bits_equal(pt, ref["pt"], "pt v%d" % variant)
        assert_bits_equal(cam.last_hit_slot, ref["slot"].to(torch.int32), "slot v%d" % variant)
        assert_bits_equal(cam.last_hit_tri, ref["tri"].to(torch.int32), "tri v%d" % variant)


def test_oracle_cuda_semantics_end_to_end(R, O, world20):
    """Oracle run with device='cuda' == the reference's real deployment (it hard-wires cuda:0): everything
    bit-exact, trig included (same libdevice)."""
    w = world20
    N = 64
    st = {k: v.cuda() for k, v in R.synth.make_env_state(w, N, seed=9).items()}
    eul = O.quat_to_euler(st["quat"])
    close(R.tensor_quat_to_eul(st["quat"]), eul, "euler", rtol=1e-6, atol=1e-7)
    pat, ci, fi = O.heightmap_pattern()
    shift = torch.tensor([0, 0, 0.0], device="cuda")
    ref = O.get_depths(st["pos"], eul, pat, w.map_indices.cuda(), w.triangles.cuda(), w.vertices.cuda(), shift)
    cam = R.Camera("cuda:0", shift, assets=(w.map_indices, w.triangles, w.vertices), sem=R.SEM_TORCH_CUDA)
    dist, pt, src = cam.get_depths(st["pos"], eul, want_hits=True)
    src_same = (bits(src.cpu()) == bits(ref["sources"].cpu())).all(2)
    assert src_same.float().mean() > 0.9999, "sources equal fraction %g" % src_same.float().mean()
    d_same = bits(dist.cpu()) == bits(ref["dist"].cpu())
    assert d_same[src_same].all(), "rays with identical sources must have identical distances"
    assert (cam.last_hit_tri.cpu().long() == ref["tri"].cpu())[src_same].all()
    rc = O.get_collisions(st["pos"], eul, st["joints"], w.rock_indices.cuda(), w.rock_triangles.cuda(), w.rock_vertices.cuda(), shift)
    rock = R.Rock_Detection("cuda:0", shift, assets=(w.rock_indices, w.rock_triangles, w.rock_vertices), sem=R.SEM_TORCH_CUDA)
    # torch-CUDA's sin / cos injected (the reference's own values on its deployment device): everything bit-identical
    wheel, body = rock.get_collisions(st["pos"], eul, st["joints"], want_collision=True, want_rays=True, trig=_trig(eul),
                                      joint_trig=joint_trig(st["joints"]))
    rays = rock.last_rays
    assert torch.equal(bits(rays[:, :, 0:3]), bits(rc["sources"])) and torch.equal(bits(rays[:, :, 3:6]), bits(rc["dirs"]))
    assert torch.equal(bits(wheel), bits(rc["wheel"])) and torch.equal(bits(body), bits(rc["body"]))
    assert torch.equal(rock.last_collision, O.check_collision(rc["wheel"], rc["body"]))
    # and with the trig injected the heightmap sources / distances / triangles of EVERY ray are bit-identical too
    dist, pt, src = cam.get_depths(st["pos"], eul, want_hits=True, trig=_trig(eul))
    assert torch.equal(bits(src), bits(ref["sources"])) and torch.equal(bits(dist), bits(ref["dist"]))
    assert torch.equal(cam.last_hit_tri.long(), ref["tri"])
    # the kernel's own sinf / cosf (no injection): rays within an ulp, distances identical wherever the rays are
    wheel, body = rock.get_collisions(st["pos"], eul, st["joints"], want_collision=True, want_rays=True)
    rays = rock.last_rays
    same = (bits(rays[:, :, 0:3]) == bits(rc["sources"])).all(2) & (bits(rays[:, :, 3:6]) == bits(rc["dirs"])).all(2)
    assert same.float().mean() > 0.99
    got = torch.cat((wheel, body), 1)
    want = torch.cat((rc["wheel"], rc["body"]), 1)
    assert (bits(got)[same] == bits(want)[same]).all()


def test_oracle_task_terms(R, O, world20):
    """calculate_metrics / is_done / Ackermann / obs against the oracle on the same device (CUDA semantics)."""
    w = world20
    N = 512
    st = {k: v.cuda() for k, v in R.synth.make_env_state(w, N, seed=21).items()}
    task = R.synth.make_task(w, st, level=2, sem=R.SEM_TORCH_CUDA)
    task.apply_actions(st["actions"])
    task.rover_rot = R.tensor_quat_to_eul(st["quat"])
    task.get_observations()
    task.calculate_metrics()
    task.is_done()
    eul = O.quat_to_euler(st["quat"])
    heading, _ = O.heading_and_dist(st["pos"], eul, st["target"])
    close(task.heading_diff, heading, "heading")
    lin, ang, lp, ap = st["actions"][:, 0], st["actions"][:, 1], st["prev_actions"][:, 0], st["prev_actions"][:, 1]
    rew, ex = O.metrics(st["pos"], st["target"], task.heading_diff, lin, lp, ang, ap, st["joints"], st["progress"],
                        task.rock_collison, 2, num_envs=N)
    close(task.rew_buf, rew, "rew_buf", rtol=1e-6, atol=1e-9)
    for k in ("pos_reward", "uprightness_penalty", "heading_contraint_penalty", "motion_contraint_penalty", "goal_angle_penalty"):
        close(task.extras[k], ex[k], k, rtol=1e-6, atol=1e-9)
    assert torch.equal(task.extras["collision_penalty"], ex["collision_penalty"])
    reset = O.is_done(st["pos"], st["target"], task.rover_rot, st["progress"], task.rock_collison, 2)
    assert torch.equal(task.reset_buf, reset)
    assert reset.sum() > 0 and reset.sum() < N
    steer, vel = O.ackermann(lin, ang)
    s2, v2 = R.Ackermann(lin, ang)
    close(s2, steer, "steer")
    close(v2, vel, "vel")
    ps, vs = O.joint_targets(steer, vel)
    close(task.joint_position_targets, ps, "position targets")
    close(task.joint_velocity_targets, vs, "velocity targets")
    stats = task.stats.cpu()
    assert stats[0] == N and stats[8] == reset.sum().item() and stats[3] == task.rock_collison.sum().item()


def test_edge_cases(R, O, world20):
    w = world20
    cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(w.map_indices, w.triangles, w.vertices), sem=R.SEM_TORCH_CPU)
    # empty batch
    d, pt, s = cam.get_depths(torch.zeros((0, 3), device="cuda"), torch.zeros((0, 3), device="cuda"))
    assert d.shape == (0, 1634) and pt.shape == (0, 1634, 3)
    # poses outside the map (cells clamp, camera.py:243), far above (all miss -> 11.0, slot 0) and upside down
    pos = torch.tensor([[-5.0, -5.0, 1.0], [30.0, 3.0, 1.0], [10.0, 10.0, 40.0], [10.0, 10.0, 0.8], [0.0, 19.99, 0.5]])
    eul = torch.tensor([[0.0, 0.0, 0.0], [0.1, -0.1, 2.0], [0.0, 0.0, 1.0], [3.1, 0.0, 0.0], [1.2, -1.2, -3.0]])
    pat, _, _ = O.heightmap_pattern()
    ref = O.get_depths(pos, eul, pat, w.map_indices, w.triangles, w.vertices, torch.tensor([0, 0, 0.0]))
    for variant in (0, 1, 2, 3):
        cam.variant = variant
        d, pt, s = cam.get_depths(pos.cuda(), eul.cuda(), trig=_trig(eul).cuda(), want_hits=True)
        assert_bits_equal(d, ref["dist"], "edge dist v%d" % variant)
        assert_bits_equal(cam.last_hit_slot, ref["slot"].to(torch.int32), "edge slot v%d" % variant)
        assert_bits_equal(pt, ref["pt"], "edge pt v%d" % variant)
    # 40 m above the ground the true hit (k ~ 39.7) loses the min against the 11.0 miss sentinel of the others
    assert (ref["dist"][2] == 11).all()
    # errors are Python exceptions, never a silent CPU path
    with pytest.raises(RuntimeError):
        cam.get_depths(pos, eul)
    with pytest.raises(RuntimeError):
        R.Ackermann(torch.zeros(4), torch.zeros(4))


def test_compact_layer_matches_full_layer(R, O, world20):
    """rvb_terrain_release_index: a heightmap layer without its K-contiguous index copy returns the same distances, hit slots,
    hit triangles and points -- including the two look-ups that went through the index (a ray whose only hit lies beyond the
    11 m miss sentinel, the hit-triangle output) -- and refuses the entry points that need the copy."""
    w = world20
    assets = (w.map_indices, w.triangles, w.vertices)
    full = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=assets)
    lean = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=assets, compact=True)
    G, K = w.map_indices.shape[1], w.map_indices.shape[0]
    assert full.layer.has_index and not lean.layer.has_index
    assert full.layer.bytes() - lean.layer.bytes() == 4 * G * G * ((K + 1) // 2 * 2)
    st = {k: v.cuda() for k, v in R.synth.make_env_state(w, 509, seed=31).items()}
    pos, eul = st["pos"].clone(), R.tensor_quat_to_eul(st["quat"]).clone()
    # envs 11 .. 45 m above the mesh (hits beyond the sentinel; camera.py:121-127 keeps the first slot <= 11.0), outside the map
    # and upside down
    pos[:40, 2] += torch.linspace(10.5, 45.0, 40, device="cuda")
    eul[:40, :2] = 0                      # level: the rays point straight down and hit inside their own cell's list
    pos[40:44] = torch.tensor([[-5.0, -5.0, 1.0], [30.0, 3.0, 1.0], [10.0, 10.0, 0.8], [0.0, 19.99, 0.5]], device="cuda")
    eul[41:44] = torch.tensor([[0.1, -0.1, 2.0], [3.1, 0.0, 0.0], [1.2, -1.2, -3.0]], device="cuda")
    for variant in (0, 3):
        full.variant = lean.variant = variant
        d0, pt0, s0 = full.get_depths(pos, eul, want_hits=True)
        slot0, tri0 = full.last_hit_slot.clone(), full.last_hit_tri.clone()
        d1, pt1, s1 = lean.get_depths(pos, eul, want_hits=True)
        assert torch.equal(bits(d0), bits(d1)) and torch.equal(bits(pt0), bits(pt1)) and torch.equal(bits(s0), bits(s1))
        assert torch.equal(slot0, lean.last_hit_slot) and torch.equal(tri0, lean.last_hit_tri)
    far = (pos[:, 2] > 20).nonzero().flatten()
    assert (d0[far] == 11).all() and (slot0[far] > 0).any()          # the far-hit walk ran and did not just return slot 0
    for variant in (1, 2):
        lean.variant = variant
        with pytest.raises(RuntimeError, match="released"):
            lean.get_depths(pos, eul)
    with pytest.raises(RuntimeError, match="released"):
        R.cast_rays(lean.layer, s0.reshape(-1, 3)[:64], s0.reshape(-1, 3)[:64])
    lean.layer.release_index()                                          # idempotent
    # the whole fused step on a compact heightmap layer
    st = R.synth.make_env_state(w, 256, seed=8, margin=3.0)
    a = R.synth.make_task(w, st, level=2)
    b = R.synth.make_task(w, st, level=2, compact_terrain=True)
    ra, rb = a.hot_step(st["actions"].cuda()), b.hot_step(st["actions"].cuda())
    assert torch.equal(ra[0], rb[0]) and torch.equal(ra[1], rb[1]) and torch.equal(ra[2], rb[2])
    assert not b.Camera.layer.has_index and b.Rock_detector.layer.has_index
    # the rock layer is built without the lists of the heightmap kernels (RVB_LAYER_INDEX_ONLY): index + two 32-byte records per triangle
    rl = b.Rock_detector.layer
    assert rl.bytes() == 4 * rl.G0 * rl.G1 * ((rl.K + 1) // 2 * 2) + 64 * rl.T


@pytest.mark.parametrize("index_only", [False, True])
def test_terrain_create_rejects_out_of_range_ids(R, world20, index_only):
    """rvb_terrain_create checks the ids on the device: a triangle id T in map_indices or a vertex id V in triangles fails the call
    with RVB_ERR_INVALID once the build kernels have run; the half-built layer is freed and the next valid layer builds."""
    w = world20
    T, V = w.triangles.shape[0], w.vertices.shape[0]
    bad_index = w.map_indices.clone()
    bad_index[-1, 3, 5] = T
    bad_tris = w.triangles.clone()
    bad_tris[T // 2, 1] = V
    shift = torch.tensor([0, 0, 0.0])
    with pytest.raises(RuntimeError, match=r"rvb_terrain_create \(map_indices holds a triangle id outside \[0,T\)\) \[status -1\]"):
        R.TerrainLayer(bad_index, w.triangles, w.vertices, shift, index_only=index_only)
    with pytest.raises(RuntimeError, match=r"rvb_terrain_create \(triangles holds a vertex id outside \[0,V\)\) \[status -1\]"):
        R.TerrainLayer(w.map_indices, bad_tris, w.vertices, shift, index_only=index_only)
    layer = R.TerrainLayer(w.map_indices, w.triangles, w.vertices, shift, index_only=index_only)
    assert layer.has_index and layer.bytes() > 0
    layer.close()


@pytest.mark.parametrize("patch,route", [(2.0, "tiles"), (4.6, "layer")])
def test_degenerate_triangles_take_the_exact_paths(R, patch, route, monkeypatch):
    """A mesh with edge-on triangles (all vertices of a patch moved onto one vertical plane: fp16 determinant 0 for a vertical ray,
    the reference's result for them is rounding noise that has to be reproduced).  The shadow kernel has no culling bound for
    them: tiles that meet more than 128 are handed to the tiled kernel (1 % of the mesh: `tiles`), a layer with more than 2 %
    goes to the tiled kernel altogether (`layer`; RVB_SHADOW_FORCE=1 keeps it on the shadow kernel, every tile over the patch
    handed back).  Always: bit-identical to the per-pair kernel."""
    w = R.synth.make_world(length=20.0, nv=200, K=64, n_stones=8, seed=5, build_index=None)
    v = w.vertices.clone()
    lo, hi = 9.0 - patch / 2, 9.0 + patch / 2
    inside = (v[:, 0].float() > lo) & (v[:, 0].float() < hi) & (v[:, 1].float() > lo) & (v[:, 1].float() < hi)
    v[inside, 0] = 9.0
    w.vertices = v
    w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device="cuda:0")
    cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(w.map_indices, w.triangles, w.vertices))
    T, ill = w.triangles.shape[0], cam.layer.unbounded_triangles
    assert (ill * 50 > T) == (route == "layer") and ill > 500, (ill, T)
    st = R.synth.make_env_state(w, 384, seed=12, margin=3.0)
    g = torch.Generator().manual_seed(3)
    st["pos"][:256, :2] = 9.0 + (torch.rand(256, 2, generator=g) - 0.5) * (patch + 4.0)          # over and around the patch
    st = {k: v_.cuda() for k, v_ in st.items()}
    eul = R.tensor_quat_to_eul(st["quat"])
    cam.variant = 1
    d1, pt1, _ = cam.get_depths(st["pos"], eul, want_hits=True)
    s1, t1 = cam.last_hit_slot.clone(), cam.last_hit_tri.clone()
    for force in (None, "1"):
        if force:
            monkeypatch.setenv("RVB_SHADOW_FORCE", force)
        cam.variant = 0
        d0, pt0, _ = cam.get_depths(st["pos"], eul, want_hits=True)
        assert torch.equal(bits(d0), bits(d1)) and torch.equal(bits(pt0), bits(pt1))
        assert torch.equal(cam.last_hit_slot, s1) and torch.equal(cam.last_hit_tri, t1)
    monkeypatch.delenv("RVB_SHADOW_FORCE", raising=False)
    assert (d1 != 11).float().mean() > 0.5


def test_full_size_properties(R, world20):
    """4096 envs: variant 0 == variant 1 bit for bit, determinism, translation of the same env set."""
    w = world20
    N = 4096
    st = {k: v.cuda() for k, v in R.synth.make_env_state(w, N, seed=77).items()}
    eul = R.tensor_quat_to_eul(st["quat"])
    cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(w.map_indices, w.triangles, w.vertices))
    d0, pt0, s0 = cam.get_depths(st["pos"], eul, want_hits=True)
    t0 = cam.last_hit_tri.clone()
    for v in (1, 2, 3):
        cam.variant = v
        d1, pt1, s1 = cam.get_depths(st["pos"], eul, want_hits=True)
        assert torch.equal(bits(d0), bits(d1)) and torch.equal(bits(pt0), bits(pt1)) and torch.equal(t0, cam.last_hit_tri)
    cam.variant = 0
    d2, _, _ = cam.get_depths(st["pos"], eul)
    assert torch.equal(bits(d0), bits(d2))
    perm = torch.randperm(N, device="cuda")
    d3, _, _ = cam.get_depths(st["pos"][perm], eul[perm])
    assert torch.equal(bits(d3), bits(d0[perm]))        # envs are independent
    assert (d0 != 11).float().mean() > 0.5


def test_knn_index_builder_matches_bruteforce(R, world20):
    """Device index builder == brute-force restatement of rover_utils.py:52-118 (ties by triangle id)."""
    w = world20
    got = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K)
    assert torch.equal(got.cpu(), w.map_indices)
    gr = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, min(w.K, w.rock_triangles.shape[0]))
    assert torch.equal(gr.cpu(), w.rock_indices[:gr.shape[0]])
    # sparse layer: 3 far-apart clusters, K larger than any cluster -> windows must grow
    g = torch.Generator().manual_seed(3)
    centers = torch.tensor([[2.0, 2.0], [17.0, 5.0], [9.0, 18.0]])
    v = (centers[:, None, :] + torch.rand(3, 90, 2, generator=g) * 0.8).reshape(-1, 2)
    v = torch.cat((v, torch.rand(v.shape[0], 1, generator=g)), 1).to(torch.float16)
    t = torch.arange(0, 270 - 2, dtype=torch.int32)
    t = torch.stack((t, t + 1, t + 2), 1)
    ref = R.synth.knn_index_bruteforce(v, t, 200, 0.1, 128)
    got = R.build_knn_index(t, v, 200, 0.1, 128)
    assert torch.equal(got.cpu(), ref)


@pytest.mark.parametrize("K", [1, 2, 37, 64, 65, 129])
def test_candidate_count_variants(R, O, world20, K):
    """Row lengths that are odd / straddle the 64-candidate chunks of the production kernel: production kernel ==
    per-pair cross-check kernel == oracle, bit for bit (distances, hit slots, hit triangles)."""
    w = world20
    idx = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, K).cpu()
    N = 48
    st = R.synth.make_env_state(w, N, seed=300 + K)
    eul = O.quat_to_euler(st["quat"])
    pat, _, _ = O.heightmap_pattern()
    ref = O.get_depths(st["pos"], eul, pat, idx, w.triangles, w.vertices, torch.tensor([0, 0, 0.0]))
    cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(idx, w.triangles, w.vertices), sem=R.SEM_TORCH_CPU)
    for variant in (0, 1, 2, 3):
        cam.variant = variant
        dist, pt, src = cam.get_depths(st["pos"].cuda(), eul.cuda(), trig=_trig(eul).cuda(), want_hits=True)
        assert_bits_equal(dist, ref["dist"], "dist K=%d v%d" % (K, variant))
        assert_bits_equal(cam.last_hit_slot, ref["slot"].to(torch.int32), "slot K=%d v%d" % (K, variant))
        assert_bits_equal(cam.last_hit_tri, ref["tri"].to(torch.int32), "tri K=%d v%d" % (K, variant))
        assert_bits_equal(pt, ref["pt"], "pt K=%d v%d" % (K, variant))


def test_far_hits_and_spread_rays(R, O, world20):
    """(a) rays whose only hits lie beyond the 11.0 miss sentinel (torch.min then returns the first slot holding
    <= 11.0, not necessarily slot 0); (b) a pattern spread over more cells than the kernel's cell histogram holds
    (falls back to one work item per ray); (c) every ray of an env in one cell (heavy cell split into items)."""
    w = world20
    cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(w.map_indices, w.triangles, w.vertices), sem=R.SEM_TORCH_CPU)
    pat, _, _ = O.heightmap_pattern()
    g = torch.Generator().manual_seed(5)
    pos = torch.cat((torch.rand(24, 2, generator=g) * 16 + 2, torch.rand(24, 1, generator=g) * 4 + 12.0), 1)     # 12 .. 16 m up, level:
    eul = torch.cat((torch.zeros(24, 2), torch.rand(24, 1, generator=g) * 6.28 - 3.14), 1)     # rays hit their own cell's nearest triangles
    pos[12:, 2] -= 2.2                                                                           # some hits on either side of 11.0
    pos = torch.cat((pos, torch.tensor([[-40.0, -40.0, 1.0], [60.0, 8.0, 1.0]])))       # all rays clamp into one edge cell / one edge row
    eul = torch.cat((eul, torch.zeros(2, 3)))
    shift = torch.tensor([0, 0, 0.0])
    ref = O.get_depths(pos, eul, pat, w.map_indices, w.triangles, w.vertices, shift)
    far = (ref["dist"] == 11) & (ref["slot"] != 0)
    for variant in (0, 1, 2, 3):
        cam.variant = variant
        d, pt, s = cam.get_depths(pos.cuda(), eul.cuda(), trig=_trig(eul).cuda(), want_hits=True)
        assert_bits_equal(d, ref["dist"], "far dist v%d" % variant)
        assert_bits_equal(cam.last_hit_slot, ref["slot"].to(torch.int32), "far slot v%d" % variant)
    assert far.any(), "the case must exercise a first-miss slot other than 0"
    # (b) a 40 m wide pattern: 4096 points on a 64 x 64 grid with 0.62 m spacing
    lin = torch.arange(64, dtype=torch.float64) * 0.62 - 19.5
    wide = torch.stack((lin[:, None].expand(64, 64).reshape(-1), lin[None, :].expand(64, 64).reshape(-1),
                        torch.full((4096,), -0.2688, dtype=torch.float64)), 1)
    pos2 = torch.tensor([[10.0, 10.0, 1.0], [3.0, 15.0, 1.2]])
    eul2 = torch.tensor([[0.05, -0.03, 0.7], [0.0, 0.1, -2.0]])
    ref2 = O.get_depths(pos2, eul2, wide, w.map_indices, w.triangles, w.vertices, shift)
    lib = R._lib.load()
    dist = torch.empty((2, 4096), dtype=torch.float16, device="cuda")
    slot = torch.empty((2, 4096), dtype=torch.int32, device="cuda")
    d_pos, d_eul, d_trig, d_pat = pos2.cuda(), eul2.cuda(), _trig(eul2).cuda(), wide.cuda()      # keep the buffers alive
    for variant in (0, 1, 2, 3):
        R._lib.check(lib.rvb_heightmap_raycast(cam.layer.handle, R._lib.ptr(d_pos), R._lib.ptr(d_eul), R._lib.ptr(d_trig),
                                               R._lib.ptr(d_pat), 4096, 2, R._lib.ptr(dist), R._lib.ptr(slot), None, None, None,
                                               None, 0, None, 0, 0, None, None, variant, None))
        torch.cuda.synchronize()
        assert_bits_equal(dist, ref2["dist"], "wide pattern dist v%d" % variant)
        assert_bits_equal(slot, ref2["slot"].to(torch.int32), "wide pattern slot v%d" % variant)


@pytest.fixture(scope="module")
def world200(R):
    """The benchmark world (BASELINE.json configs[1]): 200 x 200 m, 999 698 triangles, K = 200, index built on the device.
    fp16 coordinates up to 200 m (grid spacing 0.125 m above 128 m) are where the shadow kernel's bounds are loosest."""
    w = R.synth.make_world(length=200.0, nv=708, K=200, n_stones=2000, seed=42, build_index=None)
    w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device="cuda:0")
    return w


def test_large_world_all_variants_agree(R, world200):
    """2048 envs on the 200 m world (1 % strongly tilted, some on the map border): the production kernel (triangle
    enumeration with conservative culling) == tiled kernels == the per-pair kernel that evaluates every (ray, candidate)
    pair literally; distances, hit slots, hit triangles and intersection points bit for bit."""
    w = world200
    N = 2048
    st = R.synth.make_env_state(w, N, seed=9)
    g = torch.Generator().manual_seed(4)
    st["pos"][:64, :2] = torch.rand(64, 2, generator=g) * 6 - 3 + torch.tensor([0.0, 100.0])         # across the x = 0 border
    st["pos"][64:128, :2] = torch.rand(64, 2, generator=g) * 6 + torch.tensor([196.0, 196.0])        # around the far corner
    rp = torch.rand(128, 2, generator=g) * 2.9 - 1.45                                               # up to 83 degrees of tilt
    yaw = torch.rand(128, generator=g) * 6.28 - 3.14
    st["quat"][128:256] = R.synth.euler_to_quat_wxyz(rp[:, 0], rp[:, 1], yaw)
    st["pos"][256:288, 2] += torch.rand(32, generator=g) * 12                                       # hovering up to 12 m
    st = {k: v.cuda() for k, v in st.items()}
    eul = R.tensor_quat_to_eul(st["quat"])
    cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(w.map_indices, w.triangles, w.vertices))
    out = {}
    for v in (1, 0, 2, 3):
        cam.variant = v
        d, pt, s = cam.get_depths(st["pos"], eul, want_hits=True)
        out[v] = (d.clone(), pt.clone(), cam.last_hit_slot.clone(), cam.last_hit_tri.clone())
    for v in (0, 2, 3):
        for i, what in enumerate(("dist", "pt", "slot", "tri")):
            assert_bits_equal(out[v][i], out[1][i], "200 m world %s variant %d vs 1" % (what, v))
    assert (out[0][0] != 11).float().mean() > 0.5


def test_benchmark_world_matches_oracle(R, O, world200):
    """The ORACLE (the reference's op sequence, run on cuda:0 = the reference's own deployment) against the production kernels on
    the BENCHMARK world: 96 envs of the 200 m / 999,698-triangle terrain -- coordinates beyond 128 m (fp16 grid 0.125 m), the map
    border and corner, envs tilted up to 83 degrees, hovering envs -- heightmap distances, hit slots, hit triangles, sources,
    rock distances, collision flags, observations, rewards and reset masks.  The trigonometry is torch-CUDA's (injected), so
    every comparison is bit for bit except the fp32 reward terms (<= 1e-6 relative)."""
    w = world200
    dev = "cuda:0"
    if getattr(w, "rock_indices", None) is None:
        w.rock_indices = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, w.K, device=dev)
    N = 96
    st = R.synth.make_env_state(w, N, seed=31)
    g = torch.Generator().manual_seed(8)
    st["pos"][:24, :2] = torch.rand(24, 2, generator=g) * 70 + 129.0                                  # x, y in [129, 199]
    st["pos"][24:32, :2] = torch.rand(8, 2, generator=g) * 6 - 3 + torch.tensor([0.0, 100.0])        # across the x = 0 border
    st["pos"][32:40, :2] = torch.rand(8, 2, generator=g) * 6 + torch.tensor([196.0, 196.0])          # around the far corner
    hf = R.synth.terrain_height(w, st["pos"][:40, :2].clamp(0, 200))
    st["pos"][:40, 2] = hf + 0.5
    rp = torch.rand(16, 2, generator=g) * 2.9 - 1.45                                                 # up to 83 degrees of tilt
    st["quat"][40:56] = R.synth.euler_to_quat_wxyz(rp[:, 0], rp[:, 1], torch.rand(16, generator=g) * 6.28 - 3.14)
    st["pos"][56:64, 2] += torch.rand(8, generator=g) * 12                                           # hovering up to 12 m
    st = {k: v.to(dev) for k, v in st.items()}
    eul = O.quat_to_euler(st["quat"])
    trig = _trig(eul)
    pat, ci, fi = O.heightmap_pattern()
    shift = torch.tensor([0, 0, 0.0], device=dev)
    mi = w.map_indices.to(dev)
    ref = O.get_depths(st["pos"], eul, pat, mi, w.triangles.to(dev), w.vertices.to(dev), shift, env_chunk=8)
    cam = R.Camera(dev, shift, assets=(w.map_indices, w.triangles, w.vertices), sem=R.SEM_TORCH_CUDA)
    for variant in (0, 3):
        cam.variant = variant
        dist, pt, src = cam.get_depths(st["pos"], eul, trig=trig, want_hits=True)
        assert torch.equal(bits(src), bits(ref["sources"])), "sources v%d" % variant
        assert torch.equal(bits(dist), bits(ref["dist"])), "distances v%d" % variant
        assert torch.equal(bits(pt), bits(ref["pt"])), "intersection points v%d" % variant
        assert torch.equal(cam.last_hit_slot.long(), ref["slot"].long()), "hit slots v%d" % variant
        assert torch.equal(cam.last_hit_tri.long(), ref["tri"].long()), "hit triangles v%d" % variant
    assert (ref["dist"][:24] != 11).float().mean() > 0.5          # the far-coordinate envs do hit the terrain
    del mi
    # rock layer + collision flags
    ri = w.rock_indices.to(dev)
    rc = O.get_collisions(st["pos"], eul, st["joints"], ri, w.rock_triangles.to(dev), w.rock_vertices.to(dev), shift)
    del ri
    task = R.synth.make_task(w, {k: v.cpu() for k, v in st.items()}, device=dev, level=2, sem=R.SEM_TORCH_CUDA)
    task.parity_trig, task.parity_joint_trig = trig, joint_trig(st["joints"])
    obs, rew, reset, extras = task.hot_step(st["actions"], fused=False)
    assert torch.equal(bits(task.rock_wheel_dist), bits(rc["wheel"])) and torch.equal(bits(task.rock_body_dist), bits(rc["body"]))
    rock = O.check_collision(rc["wheel"], rc["body"])
    assert torch.equal(task.rock_collison, rock)
    lin, ang = st["actions"][:, 0], st["actions"][:, 1]
    o_obs, _, heading = O.observations(st["pos"], st["quat"], st["target"], lin, ang, ref["dist"], ci.to(dev), fi.to(dev))
    assert torch.equal(obs[:, 4:], o_obs[:, 4:]), "heightmap observation columns"
    close(obs[:, :4], o_obs[:, :4], "proprioceptive columns", rtol=1e-6, atol=1e-7)
    progress = st["progress"] + 1
    o_rew, o_ex = O.metrics(st["pos"], st["target"], task.heading_diff, lin, st["prev_actions"][:, 0], ang, st["prev_actions"][:, 1],
                            st["joints"], progress, rock, 2, num_envs=N)
    close(rew, o_rew, "rew_buf", rtol=1e-6, atol=1e-9)
    o_reset = O.is_done(st["pos"], st["target"], eul, progress, rock, 2)
    assert torch.equal(reset, o_reset)
    assert 0 < int(o_reset.sum()) < N


def test_fused_step_equals_call_sequence(R, world20):
    """The fused step (rvb_env_pre + rvb_env_post, rock layer on a forked stream) == the reference-shaped sequence of calls, for three
    consecutive steps (history shift, progress counter and statistics included); then the pipelined host front end."""
    w = world20
    N = 300
    st = R.synth.make_env_state(w, N, seed=21)
    tasks = [R.synth.make_task(w, st, device="cuda:0", level=2) for _ in range(2)]
    g = torch.Generator().manual_seed(1)
    for step in range(3):
        act = (torch.rand(N, 2, generator=g) * 2 - 1).cuda()
        outs = []
        for t, fused in zip(tasks, (True, False)):
            obs, rew, reset, extras = t.hot_step(act, fused=fused)
            torch.cuda.synchronize()
            outs.append((obs.clone(), rew.clone(), reset.clone(), t.progress_buf.clone(), t.stats.clone(), t.rock_collison.clone(),
                         t.linear_velocity.tracker.clone(), t.joint_position_targets.clone(), t.joint_velocity_targets.clone(),
                         t.heading_diff.clone(), extras["motion_contraint_penalty"].clone(), extras["collision_penalty"].clone()))
        for a, b in zip(*outs):
            assert torch.equal(a, b)
    # host pipeline: two slots, results of every step equal to the synchronous device path
    t_ref, t_pipe = tasks
    pipe = R.HostPipeline(t_pipe)
    hs = {k: v.clone() for k, v in st.items()}
    view = t_ref._rover
    slots = []
    for step in range(4):
        act = torch.rand(N, 2, generator=g) * 2 - 1
        hs["pos"][:, 0] += 0.01
        view.pos = hs["pos"].cuda()
        obs, rew, reset, _ = t_ref.hot_step(act.cuda())
        torch.cuda.synchronize()
        want = (obs.cpu().clone(), rew.cpu().clone(), reset.cpu().clone())
        k = pipe.submit(hs["pos"], hs["quat"], hs["joints"], act)
        got = pipe.result(k)
        for a, b in zip(got, want):
            assert torch.equal(a, b)


def test_packed_observation_is_lossless(R, world20):
    """rvb_step_io.obs_h16 / HostPipeline(packed_obs=True): the heightmap columns as fp16 equal the f32 columns bit for bit
    once widened, the proprioceptive columns are the same f32 values, rew / reset are unchanged."""
    w = world20
    N = 200
    st = R.synth.make_env_state(w, N, seed=33)
    t_ref = R.synth.make_task(w, st, device="cuda:0", level=2)
    t_pk = R.synth.make_task(w, st, device="cuda:0", level=2)
    pipe_ref = R.HostPipeline(t_ref)
    pipe_pk = R.HostPipeline(t_pk, packed_obs=True)
    g = torch.Generator().manual_seed(2)
    hs = {k: v.clone() for k, v in st.items()}
    for step in range(3):
        act = torch.rand(N, 2, generator=g) * 2 - 1
        hs["pos"][:, 1] += 0.02
        obs, rew, reset = pipe_ref.step(hs["pos"], hs["quat"], hs["joints"], act)
        k = pipe_pk.submit(hs["pos"], hs["quat"], hs["joints"], act)
        prop, hm16, rew2, reset2 = pipe_pk.result(k)
        assert hm16.dtype == torch.float16 and hm16.shape == (N, 1746) and prop.shape == (N, 4)
        assert torch.equal(prop, obs[:, :4]) and torch.equal(hm16.float(), obs[:, 4:])
        assert torch.equal(rew, rew2) and torch.equal(reset, reset2)
        assert torch.equal(pipe_pk.obs_f32(k), obs)
    assert pipe_pk.d2h_bytes < 0.51 * pipe_ref.d2h_bytes


def test_c3_size_step_is_shard_invariant(R, world200):
    """BASELINE.json configs[2] size (65,536 envs, big_rock_layer + stones on): the production ray-cast equals the tiled
    kernel bit for bit, and the whole fused env step gives identical obs / rew / reset / collision flags whether the envs run
    as one shard or as two (what `bench.py --gpus N` relies on: envs are independent, terrain replicated); the per-shard
    statistics add up to the single-shard ones."""
    w = world200
    if w.rock_indices is None:
        w.rock_indices = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, w.K, device="cuda:0")
    N = 65536
    st = R.synth.make_env_state(w, N, seed=77)
    whole = R.synth.make_task(w, st, device="cuda:0", level=2, num_envs_total=N)
    obs, rew, reset, _ = whole.hot_step(st["actions"].cuda())
    torch.cuda.synchronize()
    # ray-cast: shadow kernel vs tiled kernel at full size
    eul = R.tensor_quat_to_eul(st["quat"].cuda())
    cam = whole.Camera
    cam.variant = 3
    d3, _, _ = cam.get_depths(st["pos"].cuda(), eul, want_pt=False)
    cam.variant = 0
    d0, _, _ = cam.get_depths(st["pos"].cuda(), eul, want_pt=False)
    assert_bits_equal(d0, d3, "65,536 envs: shadow vs tiled")
    assert torch.equal(obs[:, 4:], (d0 * 0.5).float()[:, torch.cat((cam.heightmap.coarse_idx, cam.heightmap.fine_idx))])
    stats = torch.zeros_like(whole.stats)
    h = N // 2
    for lo, hi in ((0, h), (h, N)):
        sub = {k: v[lo:hi].contiguous() for k, v in st.items()}
        part = R.synth.make_task(w, sub, device="cuda:0", level=2, num_envs_total=N)
        o, r, z, _ = part.hot_step(sub["actions"].cuda())
        torch.cuda.synchronize()
        assert torch.equal(o, obs[lo:hi]) and torch.equal(r, rew[lo:hi]) and torch.equal(z, reset[lo:hi])
        assert torch.equal(part.rock_collison, whole.rock_collison[lo:hi])
        stats += part.stats
        del part
    assert stats[0] == N and torch.equal(stats[[0, 3, 8, 9, 10, 11, 12, 13]], whole.stats[[0, 3, 8, 9, 10, 11, 12, 13]])      # counts: exact
    assert torch.allclose(stats, whole.stats, rtol=1e-12)                                                                 # f64 sums
    assert 0 < int(whole.rock_collison.sum()) < N and 0 < int(reset.sum()) < N


@pytest.mark.parametrize("K,seed", [(200, 0), (96, 1), (255, 2)])
def test_triangle_soup_all_variants_agree(R, K, seed):
    """A mesh that is NOT a heightfield (the reference accepts any map.ply): random triangles in several overlapping layers,
    vertical walls, zero-area and collinear triangles, 10 m sheets and millimetre slivers, some far outside the map.  The
    production kernel's conservative culling must fall back to 'no bound' wherever its error model gives none: distances,
    hit slots, hit triangles and intersection points stay bit-identical to the per-pair kernel that evaluates every
    (ray, candidate) pair literally."""
    g = torch.Generator().manual_seed(100 + seed)
    L, G, T = 20.0, 200, 24000
    c = torch.rand(T, 3, generator=g) * torch.tensor([L, L, 1.5])
    size = torch.exp(torch.rand(T, 1, generator=g) * 6.0 - 5.0)                     # 7 mm .. 2.7 m
    e1 = (torch.rand(T, 3, generator=g) - 0.5) * size
    e2 = (torch.rand(T, 3, generator=g) - 0.5) * size
    kind = torch.randint(0, 10, (T,), generator=g)
    e1[kind == 0, 2] = 0.0; e2[kind == 0, 2] = 0.0                                  # horizontal sheets
    e2[kind == 1] = e1[kind == 1] * 2.0                                             # collinear (zero area)
    e2[kind == 2] = 0.0                                                             # repeated vertex
    e1[kind == 3, :2] = 0.0                                                         # vertical edge -> wall
    big = kind == 4
    e1[big] *= 10.0; e2[big] *= 10.0                                                # sheets of many metres
    c[kind == 5, :2] += 60.0                                                        # far outside the map
    v = torch.stack((c, c + e1, c + e2), 1).reshape(-1, 3).to(torch.float16)
    tri = torch.arange(3 * T, dtype=torch.int32).reshape(T, 3)
    idx = R.build_knn_index(tri, v, G, 0.1, K, device="cuda:0")
    cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(idx, tri, v))
    N = 192
    pos = torch.rand(N, 3, generator=g) * torch.tensor([L, L, 2.5]) + torch.tensor([0.0, 0.0, 0.2])
    rp = (torch.rand(N, 2, generator=g) - 0.5) * 0.6
    rp[::7] = (torch.rand(rp[::7].shape, generator=g) - 0.5) * 3.0                  # some steep / upside down
    yaw = (torch.rand(N, generator=g) - 0.5) * 6.28
    eul = torch.stack((rp[:, 0], rp[:, 1], yaw), 1)
    out = {}
    for variant in (1, 0, 3):
        cam.variant = variant
        d, pt, s = cam.get_depths(pos.cuda(), eul.cuda(), want_hits=True)
        out[variant] = (d.clone(), pt.clone(), cam.last_hit_slot.clone(), cam.last_hit_tri.clone())
    for variant in (0, 3):
        for i, what in enumerate(("dist", "pt", "slot", "tri")):
            assert_bits_equal(out[variant][i], out[1][i], "triangle soup K=%d %s variant %d vs 1" % (K, what, variant))
    hit = (out[1][0] != 11).float().mean().item()
    assert 0.05 < hit < 1.0, hit


def test_drop_in_constructors_load_reference_asset_files(R, world20, tmp_path, monkeypatch):
    """Camera(device, shift) / Rock_Detection(device, shift) without `assets` load tasks/utils/terrain/{knn_terrain,knn_rocks}/
    {map_indices,triangles,vertices}.pt relative to the CWD exactly like the reference (camera.py:154-161,
    rock_detect.py:151-158), and read_stone_info reads the reference's .npy (terrain_utils.py:416-424): results equal the
    in-memory construction."""
    import numpy as np
    w = world20
    for sub, idx, tri, ver in (("knn_terrain", w.map_indices, w.triangles, w.vertices),
                               ("knn_rocks", w.rock_indices, w.rock_triangles, w.rock_vertices)):
        d = tmp_path / "tasks" / "utils" / "terrain" / sub
        d.mkdir(parents=True)
        torch.save(idx, d / "map_indices.pt"); torch.save(tri, d / "triangles.pt"); torch.save(ver, d / "vertices.pt")
    np.save(tmp_path / "stone_info.npy", w.stone_info.numpy())
    monkeypatch.chdir(tmp_path)
    shift = torch.tensor([0, 0, 0.0])
    cam_files, cam_mem = R.Camera("cuda:0", shift), R.Camera("cuda:0", shift, assets=(w.map_indices, w.triangles, w.vertices))
    rock_files = R.Rock_Detection("cuda:0", shift)
    rock_mem = R.Rock_Detection("cuda:0", shift, assets=(w.rock_indices, w.rock_triangles, w.rock_vertices))
    st = {k: v.cuda() for k, v in R.synth.make_env_state(w, 32, seed=3).items()}
    eul = R.tensor_quat_to_eul(st["quat"])
    for a, b in zip(cam_files.get_depths(st["pos"], eul), cam_mem.get_depths(st["pos"], eul)):
        assert_bits_equal(a, b, "Camera from files vs from memory")
    assert cam_files.get_num_exteroceptive() == 1634 and cam_files.map_indices.shape == (w.G, w.G, w.K)
    for a, b in zip(rock_files.get_collisions(st["pos"], eul, st["joints"]), rock_mem.get_collisions(st["pos"], eul, st["joints"])):
        assert_bits_equal(a, b, "Rock_Detection from files vs from memory")
    s7 = R.read_stone_info(str(tmp_path / "stone_info.npy"))
    assert s7.shape == (w.stone_info.shape[0], 7) and s7.is_cuda
    assert torch.equal(s7[:, 6].cpu(), (torch.maximum(w.stone_info[:, 3], w.stone_info[:, 4]) / 4).float())


def test_reference_constructor_and_post_physics_contract(R, world20, tmp_path, monkeypatch):
    """RoverTask.from_reference(name, sim_config, env, offset) -- the reference's constructor signature (tasks/rover.py:81-87):
    numEnvs / reward scales come from sim_config.task_config, the assets from the reference's relative paths, and
    post_physics_step follows rl_task.py:239-259: progress_buf always advances, the observation / metrics / reset work only while
    env._world.is_playing(); get_states / get_extras exist."""
    import types
    w = world20
    for sub, idx, tri, ver in (("knn_terrain", w.map_indices, w.triangles, w.vertices),
                               ("knn_rocks", w.rock_indices, w.rock_triangles, w.rock_vertices)):
        d = tmp_path / "tasks" / "utils" / "terrain" / sub
        d.mkdir(parents=True)
        torch.save(idx, d / "map_indices.pt"); torch.save(tri, d / "triangles.pt"); torch.save(ver, d / "vertices.pt")
    monkeypatch.chdir(tmp_path)
    N = 48
    st = R.synth.make_env_state(w, N, seed=12)
    playing = {"on": True}
    env = types.SimpleNamespace(_world=types.SimpleNamespace(is_playing=lambda: playing["on"]))
    rewards = dict(R.rover.DEFAULT_REWARDS)
    rewards["pos_reward"] = 2.0
    sim_config = types.SimpleNamespace(config={"seed": 42}, task_config={"env": {"numEnvs": N}, "rewards": rewards})
    view = R.synth.SyntheticRoverView(st["pos"].cuda(), st["quat"].cuda(), st["joints"].cuda())
    from isaac_rover_b200.terrain_utils import stone_info_from_array
    task = R.RoverTask.from_reference("Rover", sim_config, env, None, rover_view=view,
                                      stone_info=stone_info_from_array(w.stone_info.numpy(), device="cuda:0"), heightmap=w.heightmap)
    assert task.num_envs == N and task._name == "Rover" and task.rew_scales["pos_reward"] == 2.0 and task._task_cfg is sim_config.task_config
    ref = R.synth.make_task(w, st, device="cuda:0", level=1)
    ref.rew_scales["pos_reward"] = 2.0
    task.linear_velocity.input_state(st["prev_actions"][:, 0].cuda())          # the history make_task starts from
    task.angular_velocity.input_state(st["prev_actions"][:, 1].cuda())
    for t in (task, ref):
        t.curriculum_level = 1
        t.target_positions = st["target"].cuda().clone()
        t.progress_buf = st["progress"].cuda().clone()
        t.apply_actions(st["actions"].cuda())
        t.rover_rot = R.tensor_quat_to_eul(st["quat"].cuda())
    a, b = task.post_physics_step(), ref.post_physics_step()
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])      # files + config == in-memory construction
    assert task.get_states().shape == (N, 0) and task.get_extras() is task.extras
    # paused simulation: only the step counter moves (rl_task.py:248-250)
    playing["on"] = False
    obs0, rew0, prog0 = task.obs_buf.clone(), task.rew_buf.clone(), task.progress_buf.clone()
    view.pos = view.pos + 1.0
    task.post_physics_step()
    assert torch.equal(task.progress_buf, prog0 + 1) and torch.equal(task.obs_buf, obs0) and torch.equal(task.rew_buf, rew0)
