"""CPU tests: the oracle restatement against the golden vectors the reference produced, and (only in the
container that has /root/reference) against the unmodified reference itself on fresh seeded inputs."""
import os

import pytest
import torch

import rover_oracle as O
import ref_import

HERE = os.path.dirname(os.path.abspath(__file__))
ZSHIFT = torch.tensor([0, 0, 0.0])


@pytest.fixture(scope="module")
def golden():
    return torch.load(os.path.join(HERE, "golden", "rover_golden.pt"))


def eq16(a, b):
    return torch.equal(a.view(torch.int16), b.view(torch.int16))


def test_pattern_known_answers(golden):
    pat, ci, fi = O.heightmap_pattern()
    assert pat.dtype == torch.float64 and pat.shape == (1634, 3)
    assert torch.equal(pat, golden["ref_pattern"]) and torch.equal(ci, golden["ref_coarse_idx"]) and torch.equal(fi, golden["ref_fine_idx"])
    assert len(ci) == 634 and len(fi) == 1112 and len(set(ci.tolist()) & set(fi.tolist())) == 112     # teacher_loader.py:47-48
    assert torch.equal(ci, torch.arange(634))
    assert abs(pat[:, 0].sum().item() - 1881.8) < 0.05 and abs(pat[:, 1].sum().item() + 22.4) < 0.05   # SURVEY.md section 4
    assert (pat[:, 2] == -0.2688).all()
    assert abs(pat[:, 0].min().item() - 0.15) < 1e-9 and abs(pat[:, 0].max().item() - 3.35) < 1e-9


def test_fp16_constants():
    lo = torch.zeros(1, dtype=torch.float16) - 0.1
    hi = torch.ones(1, dtype=torch.float16) + 0.1
    assert lo.item() == -0.0999755859375 and hi.item() == 1.099609375 and (hi * 10.0).item() == 11.0
    assert lo.view(torch.int16).item() & 0xFFFF == 0xAE66 and hi.view(torch.int16).item() == 0x3C66
    assert (hi * 10.0).view(torch.int16).item() == 0x4980


def test_golden_get_depths(golden):
    w = golden["world"]
    o = O.get_depths(golden["in_pos"], golden["ref_euler"], golden["ref_pattern"], w["map_indices"].to(torch.int32),
                     w["triangles"], w["vertices"], ZSHIFT)
    assert eq16(o["sources"], golden["ref_sources"]) and eq16(o["dist"], golden["ref_dist"]) and eq16(o["pt"], golden["ref_pt"])
    assert torch.equal(o["slot"].to(torch.int32), golden["oracle_slot"])


def test_golden_rocks(golden):
    w = golden["world"]
    c = O.get_collisions(golden["in_pos"], golden["ref_euler"], golden["in_joints"], w["rock_indices"].to(torch.int32),
                         w["rock_triangles"], w["rock_vertices"], ZSHIFT)
    assert eq16(c["wheel"], golden["ref_wheel"]) and eq16(c["body"], golden["ref_body"])
    assert eq16(c["sources"], golden["ref_rock_sources"]) and eq16(c["dirs"], golden["ref_rock_dirs"])
    assert torch.equal(O.check_collision(c["wheel"], c["body"]), golden["ref_rock_collision"])


def test_golden_ray_distance(golden):
    k, pt = O.ray_distance(golden["in_rd_src"], golden["in_rd_dir"], golden["in_rd_tri"])
    assert eq16(k, golden["ref_rd_k"]) and eq16(pt, golden["ref_rd_pt"])
    assert k.tolist()[:5] == [1.0, -1.0, 11.0, 11.0, 11.0]          # above, below (negative kept), outside, degenerate, parallel
    k, pt = O.ray_distance(golden["in_rr_src"], golden["in_rr_dir"], golden["in_rr_tri"])
    assert eq16(k, golden["ref_rr_k"]) and eq16(pt, golden["ref_rr_pt"])


def test_golden_task_terms(golden):
    g = golden
    assert torch.equal(O.quat_to_euler(g["in_quat"]), g["ref_euler"])
    steer, vel = O.ackermann(g["in_actions"][:, 0], g["in_actions"][:, 1])
    assert torch.equal(steer, g["ref_steer"]) and torch.equal(vel, g["ref_vel"])
    steer, vel = O.ackermann(g["in_ka_lin"], g["in_ka_ang"])
    assert torch.equal(steer, g["ref_ka_steer"]) and torch.equal(vel, g["ref_ka_vel"])
    assert torch.allclose(steer[0], torch.tensor([0.20421, 0.15067, 0, 0, -0.19193, -0.14151]), atol=1e-5)
    assert torch.allclose(vel[1], torch.tensor([5.8315, -5.8315, 4.47, -4.47, 5.6316, -5.6316]), atol=1e-4)
    assert (vel[2] == 5.0).all() and (vel[3] == 0).all()
    lin, ang = g["in_actions"][:, 0], g["in_actions"][:, 1]
    obs, eul, heading = O.observations(g["in_pos"], g["in_quat"], g["in_target"], lin, ang, g["ref_dist"],
                                       g["ref_coarse_idx"], g["ref_fine_idx"])
    assert torch.equal(obs, g["ref_obs"]) and torch.equal(heading, g["ref_heading"])
    rew, ex = O.metrics(g["in_pos"], g["in_target"], heading, lin, g["in_prev_actions"][:, 0], ang, g["in_prev_actions"][:, 1],
                        g["in_joints"], g["in_progress"], g["ref_rock_collision"], 2)
    assert torch.equal(rew, g["ref_rew"])
    for k, v in g["ref_extras"].items():
        assert torch.equal(ex[k], v), k
    assert torch.equal(O.is_done(g["in_pos"], g["in_target"], eul, g["in_progress"], g["ref_rock_collision"], 2), g["ref_reset"])
    rew1, _ = O.metrics(g["in_pos"], g["in_target"], heading, lin, g["in_prev_actions"][:, 0], ang, g["in_prev_actions"][:, 1],
                        g["in_joints"], g["in_progress"], None, 1)
    assert torch.equal(rew1, g["ref_rew_level1"])
    assert torch.equal(O.is_done(g["in_pos"], g["in_target"], eul, g["in_progress"], None, 1), g["ref_reset_level1"])


def test_golden_stones(golden):
    g = golden
    s7 = O.read_stone_info(g["world"]["stone_info6"].numpy())
    assert torch.equal(s7, g["ref_stone7"])
    assert torch.equal(O.nearest_stone_edge(g["in_target"][:, 0:2], s7), g["ref_goal_nearest"])
    assert int(O.goal_invalid(g["in_target"][:, 0:2], s7).sum()) == g["ref_goal_count"]
    moved = O.avoid_pos_rock_collision(g["in_spawn_pos"], s7)
    assert torch.equal(moved, g["ref_spawn_pos"])
    assert torch.equal(O.pos_height(g["world"]["heightmap"], moved[:, 0:2], g["world"]["hm_res"], 1, torch.tensor([0.0, 0.0])),
                       g["ref_spawn_height"])


# ------------------------------------------------------------------ against the reference itself (CPU container only)
needs_ref = pytest.mark.skipif(not ref_import.available(), reason="reference tree not present (GPU box)")


@needs_ref
@pytest.mark.reference
def test_oracle_matches_reference_fresh_world():
    import isaac_rover_b200
    from isaac_rover_b200 import synth
    import ref_world
    ns = ref_import.load("cpu")
    world = synth.make_world(length=10.0, nv=36, K=64, n_stones=6, seed=123)
    st = synth.make_env_state(world, 12, seed=5, margin=3.0)
    fake = ref_world.make_fake_task(ns, world, st, level=2)
    eul = ns.tensor_quat_to_eul(st["quat"])
    assert torch.equal(O.quat_to_euler(st["quat"]), eul)
    pat, ci, fi = O.heightmap_pattern()
    d, pt, src = fake.Camera.get_depths(st["pos"], eul)
    o = O.get_depths(st["pos"], eul, pat, world.map_indices, world.triangles, world.vertices, ZSHIFT)
    assert eq16(o["dist"], d) and eq16(o["pt"], pt) and eq16(o["sources"], src)
    wd, bd = fake.Rock_detector.get_collisions(st["pos"], eul, st["joints"])
    c = O.get_collisions(st["pos"], eul, st["joints"], world.rock_indices, world.rock_triangles, world.rock_vertices, ZSHIFT)
    assert eq16(c["wheel"], wd) and eq16(c["body"], bd)
    RT = ns.RoverTask
    RT.get_observations(fake)
    lin, ang = st["actions"][:, 0], st["actions"][:, 1]
    obs, _, heading = O.observations(st["pos"], st["quat"], st["target"], lin, ang, d, ci, fi)
    assert torch.equal(obs, fake.obs_buf)
    RT.calculate_metrics(fake)
    RT.is_done(fake)
    rew, ex = O.metrics(st["pos"], st["target"], heading, lin, st["prev_actions"][:, 0], ang, st["prev_actions"][:, 1],
                        st["joints"], st["progress"], fake.rock_collison, 2)
    assert torch.equal(rew, fake.rew_buf)
    assert torch.equal(O.is_done(st["pos"], st["target"], eul, st["progress"], fake.rock_collison, 2), fake.reset_buf)
    steer, vel = ns.Ackermann(lin, ang, "cpu")
    s2, v2 = O.ackermann(lin, ang)
    assert torch.equal(s2, steer) and torch.equal(v2, vel)


def test_product_pattern_matches_reference(golden):
    """The product's pattern against the reference Heightmap's distribution / coarse_idx / fine_idx, as make_golden.py stored
    them."""
    import isaac_rover_b200  # noqa: F401
    from isaac_rover_b200.heightmap_distribution import build_pattern
    pts, ci, fi = build_pattern()
    assert torch.equal(torch.from_numpy(pts), golden["ref_pattern"])
    assert torch.equal(torch.from_numpy(ci), golden["ref_coarse_idx"]) and torch.equal(torch.from_numpy(fi), golden["ref_fine_idx"])


def test_golden_spawn_direct_path():
    """cdist's direct path (<= 25 rows on both sides): the oracle reproduces the reference's spawn loop and nearest stone edge bit
    for bit on the vectors tests/golden/make_spawn_golden.py took from the reference."""
    sg = torch.load(os.path.join(HERE, "golden", "spawn_direct_golden.pt"))
    assert len(sg["cases"]) == 4
    for case in sg["cases"]:
        assert case["in_pos"].shape[0] <= 25 and case["stone7"].shape[0] <= 25
        assert torch.equal(O.avoid_pos_rock_collision(case["in_pos"].clone(), case["stone7"]), case["ref_pos"])
        assert torch.equal(O.nearest_stone_edge(case["in_pos"][:, 0:2], case["stone7"]), case["ref_nearest"])
