"""The policy tensor-core probes (tests/policy_probe.py) checked without a GPU: the exact probes' construction holds, their
fp64 answer is what fp32 gives in any order, the emulated tensor-core arithmetic reproduces it, every emulated kernel
defect changes at least one probe output, and the dense sweep's statistical gate tells fp32-grade from TF32-grade."""
import pytest
import torch

import policy_oracle as PO
import policy_probe as PP

CASES = PP.probe_cases()


@pytest.fixture(scope="module")
def probes():
    return {name: PP.make_exact_probe(**kw) for name, kw in CASES.items()}


def test_generator_invariants(probes):
    """make_exact_probe asserts invariants 1-5 itself; here: the probes carry what the GPU test relies on."""
    for name, pr in probes.items():
        for k, v in pr.sd.items():
            assert torch.equal(PP.tf32(v), v), (name, k)                        # every parameter is a tf32 number
        assert pr.act in PP.EXACT_ACTS
        assert torch.equal(pr.pre.to(torch.float32).double(), pr.pre), name    # the head's sum is an fp32 number
        if not pr.tanh:
            assert torch.equal(pr.expected.double(), pr.pre), name
        assert bool((pr.expected != 0).any()), name
    # about half of the fine observation values carry a lo part; coarse ones never do
    obs = probes["dense_all_fine"].obs[:, PP.P:]
    lo = PP.split(obs)[1] != 0
    assert 0.3 < lo.double().mean().item() < 0.7
    one = probes["lo_row127_d_last"].obs
    rows, cols = torch.nonzero(PP.split(one[:, PP.P:])[1]).T
    assert set(rows.tolist()) == {127} and set((cols + PP.P).tolist()) <= {PP.P + 634 + 1110, PP.P + 634 + 1111}
    # a broken invariant is refused, not silently accepted
    with pytest.raises(AssertionError):
        PP.make_exact_probe(act="elu")
    bad = PP.probe_obs(4, 634, 1112, seed=0)
    bad[1, 10] = 1.0 + 2.0 ** -23                                               # 24 significant bits
    with pytest.raises(AssertionError):
        PP.make_exact_probe(obs=bad)


def test_required_coverage(probes):
    """Paths through the proprio columns, both halves of the 256-wide layer, features 128-159 of the 160-wide one, every
    head output; lo parts in single rows 0, 127 and 129 (last live row of a ragged tile); a 65-chunk encoder."""
    paths = [p for pr in probes.values() for p in pr.paths]
    assert {0, 1, 2, 3} <= {p[0] for p in paths}
    assert any(p[1] >= 128 for p in paths) and any(p[1] < 128 for p in paths)
    assert any(128 <= p[2] < 160 for p in paths)
    assert {0, 1, 2, 3} == {p[4] for p in probes["dense_all_fine"].paths}
    assert {pr.n_head for pr in probes.values()} == {1, 2, 3, 4}
    assert max(pr.D for pr in probes.values()) > 64 * 32


def _reversed(sd):
    """The same network with every layer's inputs in reverse order (observation slices reversed by the caller; every hidden
    layer's outputs reversed, and the next layer's columns with them; the concat reversed block by block)."""
    W = {n: sd[PP.KEYS[n] + ".weight"].clone() for n in PP.KEYS}
    B = {n: sd[PP.KEYS[n] + ".bias"].clone() for n in PP.KEYS}
    W["es1"], W["ed1"] = W["es1"].flip(1), W["ed1"].flip(1)
    for prev, nxt in (("es1", "es2"), ("ed1", "ed2"), ("m1", "m2"), ("m2", "m3"), ("m3", "head")):
        W[prev], B[prev], W[nxt] = W[prev].flip(0), B[prev].flip(0), W[nxt].flip(1)
    for enc, c in (("es2", slice(PP.P, PP.P + 60)), ("ed2", slice(PP.P + 60, PP.P + 120))):
        W[enc], B[enc] = W[enc].flip(0), B[enc].flip(0)
        W["m1"][:, c] = W["m1"][:, c].flip(1)
    out = {}
    for n in PP.KEYS:
        out[PP.KEYS[n] + ".weight"], out[PP.KEYS[n] + ".bias"] = W[n], B[n]
    return out


def test_fp64_answer_equals_fp32_in_two_orders(probes):
    """Exactness: torch fp32 (its own blocked order), fp32 in reversed feature order and fp32 on one thread all give the fp64
    answer."""
    threads = torch.get_num_threads()
    for name, pr in probes.items():
        a = PO.forward(pr.sd, pr.obs, PP.P, pr.S, pr.D, pr.act, actor=False, dtype=torch.float32)
        assert torch.equal(a.double(), pr.pre), name
        obs = torch.cat((pr.obs[:, :PP.P], pr.obs[:, PP.P:PP.P + pr.S].flip(1), pr.obs[:, PP.P + pr.S:].flip(1)), 1)
        b = PO.forward(_reversed(pr.sd), obs, PP.P, pr.S, pr.D, pr.act, actor=False, dtype=torch.float32)
        assert torch.equal(b.double(), pr.pre), name
        # and with one thread (another blocking of the matmuls)
        torch.set_num_threads(1)
        try:
            b = PO.forward(pr.sd, pr.obs, PP.P, pr.S, pr.D, pr.act, actor=False, dtype=torch.float32)
        finally:
            torch.set_num_threads(threads)
        assert torch.equal(b.double(), pr.pre), name


def test_emulation_is_exact_on_every_probe(probes):
    for name, pr in probes.items():
        got = PP.emulate_tc(pr.sd, pr.obs, pr.S, pr.D, pr.act, pr.tanh)
        assert torch.equal(got, pr.expected), name
    pr = probes["dense_all_fine"]                                             # any accumulator rounding: exact too
    assert torch.equal(PP.emulate_tc(pr.sd, pr.obs, pr.S, pr.D, pr.act, pr.tanh, acc="rz"), pr.expected)


def _detected(probes, **mutation):
    for pr in probes.values():
        got = PP.emulate_tc(pr.sd, pr.obs, pr.S, pr.D, pr.act, pr.tanh, **mutation)
        if not torch.equal(got, pr.expected):
            return True
    return False


@pytest.mark.parametrize("mutation", [
    dict(drop_lo="all"), dict(single=True), dict(skip_row=127),
    dict(swap=("es1", 32)), dict(swap=("ed1", 1088)), dict(swap=("m1", 32)), dict(swap=("m1", 64)), dict(swap=("m1", 96)),
    dict(swap=("m2", 128)), dict(swap=("m3", 32))], ids=str)
def test_every_mutation_is_caught(probes, mutation):
    assert _detected(probes, **mutation)


def test_dropping_the_lo_mma_of_any_one_chunk_is_caught(probes):
    """Every first-layer chunk of both encoders (the last one partial), at the shipped split and at a 65-chunk encoder."""
    small = {k: v for k, v in probes.items() if k in ("dense_all_fine", "head1")}
    for enc, n in (("s", 634), ("d", 1112)):
        for c in range((n + 31) // 32):
            assert _detected(small, drop_lo=(enc, c)), (enc, c)
    wide = {"aliased_chunks": probes["aliased_chunks"]}
    for c in (0, 1, 63, 64):
        assert _detected(wide, drop_lo=("d", c)), c
    only64 = {"lo_chunk64_only": probes["lo_chunk64_only"]}
    assert _detected(only64, drop_lo=("d", 64)) and not _detected(only64, drop_lo=("d", 0))


def _dense_case(S, D, N, act, seed, obs_kind="fp32"):
    torch.manual_seed(seed)
    sd = {}
    for name, (i, o) in {"es1": (S, 80), "es2": (80, 60), "ed1": (D, 80), "ed2": (80, 60), "m1": (124, 256), "m2": (256, 160),
                         "m3": (160, 128), "head": (128, 2)}.items():
        bd = 1 / i ** 0.5
        sd[PP.KEYS[name] + ".weight"] = (torch.rand(o, i) * 2 - 1) * bd
        sd[PP.KEYS[name] + ".bias"] = (torch.rand(o) * 2 - 1) * bd
    obs = torch.rand(N, PP.P + S + D) * 2 - 0.5
    if obs_kind == "fp16":
        obs[:, PP.P:] = (obs[:, PP.P:] * 5.5).half().float()
    return sd, obs


@pytest.mark.parametrize("act", ["leakyrelu", "relu", "tanh"])
def test_statistical_gate_tells_fp32_grade_from_tf32(act):
    """The GPU sweep's gate (policy_probe.fp32_gate) on emulated arithmetic: the kernel's arithmetic passes, a kernel
    that never issues the first layers' lo MMAs or that runs single-pass TF32 fails."""
    S, D = 634, 1112
    for kind in ("fp32", "fp16"):
        sd, obs = _dense_case(S, D, 1000, act, 7, kind)
        for tanh in (False, True):
            ref = PO.forward(sd, obs, PP.P, S, D, act, actor=tanh, dtype=torch.float64)
            gate = PP.fp32_gate(PP.max_abs_err(PO.forward(sd, obs, PP.P, S, D, act, actor=tanh), ref))
            assert PP.max_abs_err(PP.emulate_tc(sd, obs, S, D, act, tanh), ref) <= gate
            assert PP.max_abs_err(PP.emulate_tc(sd, obs, S, D, act, tanh, single=True), ref) > gate
            if kind == "fp32":                         # fp16-valued observations have no lo part to drop
                assert PP.max_abs_err(PP.emulate_tc(sd, obs, S, D, act, tanh, drop_lo="all"), ref) > gate
