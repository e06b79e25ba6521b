"""GPU parity of the policy-inference epilogue (SURVEY.md 8f-3): rvb_policy_forward through the reference-named mirror
(isaac_rover_2.0_b200/model.py) against (a) the outputs the UNMODIFIED reference models produced (tests/golden/
policy_golden.pt) and (b) oracle/policy_oracle.py in fp64.

Tolerance: 2e-5 absolute on tanh(mean) in [-1, 1] and on the value (|v| < 1 here).  The reference computes fp32 nn.Linear;
the kernel is an fp32 FMA chain with another summation order, so bit-exactness is not defined (torch-CPU and torch-CUDA
disagree with each other at this level too).
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
TOL = 2e-5


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import isaac_rover_b200
    return isaac_rover_b200


@pytest.fixture(scope="module")
def PO():
    import policy_oracle
    return policy_oracle


@pytest.fixture(scope="module")
def golden():
    return torch.load(os.path.join(HERE, "golden", "policy_golden.pt"))["leakyrelu"]


def _models(R, S=634, D=1112, act="leakyrelu", p=4):
    net = R.model.NetworkInfo([256, 160, 128], [80, 60], [80, 60], [80, 60], act)
    info = R.model.ObserverationInfo(p, S, D, 0)
    actor = R.model.StochasticActorHeightmap(p + S + D, 2, net, info, device="cuda:0")
    critic = R.model.DeterministicHeightmap(p + S + D, 2, net, info, device="cuda:0")
    return actor, critic


def test_golden_reference_outputs(R, golden):
    actor, critic = _models(R)
    actor.load_state_dict(golden["actor_sd"])
    critic.load_state_dict(golden["critic_sd"])
    obs = golden["obs"].cuda()
    mean, log_std = actor.compute(obs, None, "policy")
    value = critic.compute(obs, None, "value")
    assert mean.shape == (70, 2) and value.shape == (70, 1) and mean.dtype == torch.float32
    assert torch.equal(log_std.cpu(), golden["log_std"])
    assert (mean.cpu() - golden["mean"]).abs().max().item() < TOL
    assert (value.cpu() - golden["value"]).abs().max().item() < TOL
    # state_dict round trip keeps the reference's keys and values
    sd = actor.state_dict()
    assert set(sd) == set(golden["actor_sd"])
    assert all(torch.equal(sd[k], golden["actor_sd"][k]) for k in sd)


@pytest.mark.parametrize("act", ["leakyrelu", "relu", "elu", "tanh", "sigmoid", "relu6"])
@pytest.mark.parametrize("N,S,D,p", [(1, 634, 1112, 4), (31, 137, 203, 4), (97, 33, 1, 0), (64, 273 - 100, 100, 8)])
def test_against_fp64_oracle(R, PO, act, N, S, D, p):
    torch.manual_seed(1000 + N)
    actor, critic = _models(R, S, D, act, p)                       # nn.Linear-style random initialisation
    obs = (torch.rand(N, p + S + D) * 2 - 0.5)
    obs_d = obs.cuda()
    mean, _ = actor.compute(obs_d)
    value = critic.compute(obs_d)
    mean64 = PO.forward(actor.state_dict(), obs, p, S, D, act, actor=True, dtype=torch.float64)
    value64 = PO.forward(critic.state_dict(), obs, p, S, D, act, actor=False, dtype=torch.float64)
    assert (mean.cpu().double() - mean64).abs().max().item() < TOL
    assert (value.cpu().double() - value64).abs().max().item() < TOL * max(1.0, value64.abs().max().item())


def test_strided_rows_and_determinism(R, PO):
    """obs_buf may be a view of a wider buffer (row stride > columns); two calls give identical bits; env order is free."""
    torch.manual_seed(5)
    actor, _ = _models(R)
    wide = torch.rand(300, 1800, device="cuda")
    obs = wide[:, :1750]
    a = actor.compute(obs)[0]
    b = actor.compute(obs)[0]
    c = actor.compute(obs.contiguous())[0]
    assert torch.equal(a, b) and torch.equal(a, c)
    perm = torch.randperm(300, device="cuda")
    d = actor.compute(obs[perm].contiguous())[0]
    assert torch.equal(d, a[perm])
    ref = PO.forward(actor.state_dict(), obs.cpu(), 4, 634, 1112, "leakyrelu", actor=True, dtype=torch.float64)
    assert (a.cpu().double() - ref).abs().max().item() < TOL


def test_consumes_the_step_observation(R, PO):
    """End of the chain: the fused env step writes obs_buf, the policy reads it in place (the call order of the reference's
    trainer: env.step -> policy.compute(states))."""
    dev = "cuda:0"
    w = R.synth.make_world(length=12.0, nv=44, K=64, n_stones=8, seed=3, build_index=None)
    w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device=dev).cpu()
    kr = min(w.K, w.rock_triangles.shape[0])
    w.rock_indices = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, kr, device=dev).cpu()
    st = R.synth.make_env_state(w, 70, seed=5, margin=3.0)
    task = R.synth.make_task(w, st, device=dev, level=2)
    obs, rew, reset, extras = task.hot_step(st["actions"].to(dev))
    assert obs.shape == (70, 1750)
    torch.manual_seed(9)
    actor, critic = _models(R)
    mean, _ = actor.compute(obs)
    value = critic.compute(obs)
    mean64 = PO.forward(actor.state_dict(), obs.cpu(), 4, 634, 1112, "leakyrelu", actor=True, dtype=torch.float64)
    value64 = PO.forward(critic.state_dict(), obs.cpu(), 4, 634, 1112, "leakyrelu", actor=False, dtype=torch.float64)
    assert (mean.cpu().double() - mean64).abs().max().item() < TOL
    assert (value.cpu().double() - value64).abs().max().item() < TOL * max(1.0, value64.abs().max().item())


def test_pair_launch_equals_single_launches(R):
    """rvb_policy_forward_pair (actor + critic in one grid) returns the very bits of the two single launches."""
    torch.manual_seed(21)
    actor, critic = _models(R)
    for N in (1, 33, 4096):
        obs = torch.rand(N, 1750, device="cuda")
        mean, value = R.model.compute_pair(actor, critic, obs)
        assert torch.equal(mean, actor.compute(obs)[0]) and torch.equal(value, critic.compute(obs))
        assert mean.shape == (N, 2) and value.shape == (N, 1)
    with pytest.raises(RuntimeError):
        R.model.compute_pair(actor, critic, torch.zeros(3, 1750))


def test_tensor_core_and_ffma2_paths_agree(R):
    """rvb_policy_variant: 2 (default: the network on tcgen05 with tf32 hi + lo operands, accumulators in TMEM) sums in another
    order than 1 (the packed FFMA2 kernel for every shape) and stays within 1e-5 of it -- on arbitrary fp32 observations (three
    MMAs per k-step) and on fp16-valued ones like the step's obs_buf (the A operand is exact in tf32: two MMAs per k-step).
    On the FFMA2 path the one-network launch returns the very bits of the pair launch."""
    lib = R._lib.load()
    torch.manual_seed(8)
    actor, critic = _models(R)
    obs = torch.rand(1000, 1750, device="cuda")
    assert lib.rvb_policy_variant(-1) == 2                            # default: the whole network on tcgen05
    try:
        m2, v2 = R.model.compute_pair(actor, critic, obs)
        s2 = actor.compute(obs)[0]
        assert lib.rvb_policy_variant(1) == 2
        m1, v1 = R.model.compute_pair(actor, critic, obs)
        s1 = actor.compute(obs)[0]
        obs16 = obs.clone()
        obs16[:, 4:] = (obs[:, 4:] * 5.5).half().float()              # what the ray-cast writes: fp16 values in f32 columns
        m1h, v1h = R.model.compute_pair(actor, critic, obs16)
        assert lib.rvb_policy_variant(2) == 1
        m2h, v2h = R.model.compute_pair(actor, critic, obs16)
    finally:
        lib.rvb_policy_variant(2)
    assert torch.equal(s1, m1)
    for a, b in ((m2, m1), (v2, v1), (s2, m1), (m2h, m1h), (v2h, v1h)):
        assert (a - b).abs().max().item() <= 1e-5, (a - b).abs().max().item()
    # ragged tile counts of the 128-env tensor-core tiles
    for n in (1, 127, 129, 300):
        lib.rvb_policy_variant(1)
        ref = R.model.compute_pair(actor, critic, obs16[:n])
        lib.rvb_policy_variant(2)
        got = R.model.compute_pair(actor, critic, obs16[:n])
        assert (got[0] - ref[0]).abs().max().item() <= 1e-5 and (got[1] - ref[1]).abs().max().item() <= 1e-5
    lib.rvb_policy_variant(2)
    big = torch.rand(2048 + 77, 1750, device="cuda")                 # the default dispatch is the tensor-core path
    big[:, 4:] = (big[:, 4:] * 5.5).half().float()
    got = R.model.compute_pair(actor, critic, big)
    lib.rvb_policy_variant(1)
    ref = R.model.compute_pair(actor, critic, big)
    lib.rvb_policy_variant(2)
    assert (got[0] - ref[0]).abs().max().item() <= 1e-5 and (got[1] - ref[1]).abs().max().item() <= 1e-5
    assert not torch.equal(got[0], ref[0])                             # ... and it really is another summation order


def test_argument_validation(R):
    actor, _ = _models(R)
    with pytest.raises(RuntimeError):
        actor.compute(torch.zeros(4, 1750))                         # CPU tensor: no CPU path
    with pytest.raises(RuntimeError):
        actor.compute(torch.zeros(4, 100, device="cuda"))           # rows shorter than the network input
    net = R.model.NetworkInfo([256, 160, 64], [80, 60], [80, 60], [80, 60], "leakyrelu")
    with pytest.raises(RuntimeError):                               # widths other than the reference's: RVB_ERR_UNSUPPORTED
        R.model.StochasticActorHeightmap(1750, 2, net, R.model.ObserverationInfo(4, 634, 1112, 0), device="cuda:0")
    empty = actor.compute(torch.zeros(0, 1750, device="cuda"))[0]
    assert empty.shape == (0, 2)


def test_throughput_note(R):
    """Not a gate: prints the kernel time at the benchmark size so the round's log carries a first number."""
    actor, _ = _models(R)
    obs = torch.rand(4096, 1750, device="cuda")
    for _ in range(3):
        actor.compute(obs)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(20):
        actor.compute(obs)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20
    print("\npolicy_forward 4096 envs: %.4f ms/launch (%.1f M envs/s)" % (ms, 4096 / ms / 1e3))
    assert ms > 0
    big = torch.rand(65536, 1750, device="cuda")
    _, critic = _models(R)
    for _ in range(2):
        R.model.compute_pair(actor, critic, big)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(5):
        R.model.compute_pair(actor, critic, big)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    lib = R._lib.load()
    lib.rvb_policy_variant(1)
    try:
        for _ in range(2):
            R.model.compute_pair(actor, critic, big)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            R.model.compute_pair(actor, critic, big)
        e1.record()
        torch.cuda.synchronize()
    finally:
        lib.rvb_policy_variant(2)
    print("policy_forward_pair 65536 envs, FFMA2 kernel: %.4f ms/launch" % (e0.elapsed_time(e1) / 5))
    print("policy_forward_pair 65536 envs: %.4f ms/launch (%.1f M envs/s, %.1f fp32 TFLOP/s)" % (
        ms, 65536 / ms / 1e3, 2 * 2 * 65536 * 243.3e3 / ms / 1e9))
