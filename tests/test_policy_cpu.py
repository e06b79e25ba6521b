"""Policy-epilogue oracle (oracle/policy_oracle.py) pinned against the UNMODIFIED reference models and the golden fixture."""
import importlib.util
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import policy_oracle, ref_import  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "policy_golden.pt")
GOLDEN_THREADS = 8


def _gen():
    spec = importlib.util.spec_from_file_location("make_policy_golden", os.path.join(ROOT, "tests", "golden", "make_policy_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_golden_fixture_matches_oracle_bit_for_bit():
    """The fixture was computed by torch's fp32 CPU matmul on GOLDEN_THREADS threads; the CPU BLAS splits the work by thread
    count, so the same bits come out only with that count."""
    g = torch.load(GOLDEN)["leakyrelu"]
    threads = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        mean = policy_oracle.forward(g["actor_sd"], g["obs"], 4, 634, 1112, "leakyrelu", actor=True)
        value = policy_oracle.forward(g["critic_sd"], g["obs"], 4, 634, 1112, "leakyrelu", actor=False)
    finally:
        torch.set_num_threads(threads)
    assert mean.shape == (70, 2) and value.shape == (70, 1)
    assert torch.equal(mean, g["mean"]) and torch.equal(value, g["value"])
    assert torch.equal(g["log_std"], torch.zeros(2))                       # model.py:178
    # the fp32 path is itself within the GPU gate's tolerance of exact arithmetic
    mean64 = policy_oracle.forward(g["actor_sd"], g["obs"], 4, 634, 1112, "leakyrelu", actor=True, dtype=torch.float64)
    assert (mean.double() - mean64).abs().max() < 2e-5


@pytest.mark.skipif(not ref_import.available(), reason="reference tree not present")
@pytest.mark.parametrize("activation", ["leakyrelu", "relu", "elu", "tanh", "sigmoid", "relu6"])
def test_oracle_matches_reference_models(activation):
    gen = _gen()
    S, D = (634, 1112) if activation == "leakyrelu" else (137, 203)        # the C5 patterns change the split
    actor, critic = gen.reference_models(num_obs=4 + S + D, num_sparse=S, num_dense=D, activation=activation, seed=3)
    obs = gen.synthetic_obs(33, 4 + S + D, seed=5)
    with torch.no_grad():
        mean_ref, _ = actor.compute(obs, None, "policy")
        value_ref = critic.compute(obs, None, "value")
    mean = policy_oracle.forward(gen.state_dict_of(actor), obs, 4, S, D, activation, actor=True)
    value = policy_oracle.forward(gen.state_dict_of(critic), obs, 4, S, D, activation, actor=False)
    assert torch.equal(mean, mean_ref) and torch.equal(value, value_ref)


def test_reference_state_dict_keys():
    g = torch.load(GOLDEN)["leakyrelu"]
    keys = set(g["actor_sd"])
    for k in ("encoder0.encoder.0.layer.0.weight", "encoder0.encoder.1.layer.0.bias", "encoder1.encoder.0.layer.0.weight",
              "network.0.layer.0.weight", "network.2.layer.0.bias", "network.3.weight", "network.3.bias", "log_std_parameter"):
        assert k in keys, k
    assert g["actor_sd"]["encoder0.encoder.0.layer.0.weight"].shape == (80, 634)      # teacher_loader.py:47-48 sizes
    assert g["actor_sd"]["encoder1.encoder.0.layer.0.weight"].shape == (80, 1112)
    assert g["actor_sd"]["network.0.layer.0.weight"].shape == (256, 124)
    assert g["critic_sd"]["network.3.weight"].shape == (1, 128)


def test_policy_has_no_cpu_path():
    import isaac_rover_b200 as R
    net = R.model.NetworkInfo([256, 160, 128], [80, 60], [80, 60], [80, 60], "leakyrelu")
    info = R.model.ObserverationInfo(4, 634, 1112, 0)
    with pytest.raises(RuntimeError):
        R.model.StochasticActorHeightmap(1750, 2, net, info, device="cpu")
