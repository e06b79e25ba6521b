"""The policy network's tensor-core path (policy_l1_tc_kernel + policy_tail_tc_kernel) held to an fp64 oracle.

1. Which kernel ran: every case names the kernels a torch.profiler trace shows.
2. Exact probes (tests/policy_probe.py): networks and observations on which fp32 arithmetic in any order is exact; both
   paths, single and pair launches, must return the probe's answer bit for bit (the actor: within the 2 ulp CUDA
   documents for tanhf, and the two paths bit-identical).
3. Dense random sweep against fp64: gate err <= max(32 x err_fp32, 1e-7), err_fp32 = the error of torch fp32 on the same
   device with TF32 matmuls off.  Every case's errors are printed (pytest -rP shows them).
4. Pipeline cases: the fused step's observations after the noise hook, the benchmark's 131,072 rows, and 320,000 rows
   whose observations pass 2^31 bytes.
"""
import math

import pytest
import torch

import policy_oracle as PO
import policy_probe as PP

pytestmark = pytest.mark.gpu

TC = {"policy_l1_tc_kernel", "policy_tail_tc_kernel"}
FFMA = {"policy_forward_kernel"}


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import isaac_rover_b200
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield isaac_rover_b200
    torch.backends.cuda.matmul.allow_tf32 = prev
    isaac_rover_b200._lib.load().rvb_policy_variant(2)


@pytest.fixture(scope="module")
def table():
    rows = []
    yield rows
    if rows:
        print("\n%-44s %10s %10s %10s %10s" % ("case", "TC", "FFMA2", "fp32", "gate"))
        for r in rows:
            print("%-44s %10.2e %10.2e %10.2e %10.2e" % r)


def _record(table, row):
    print("%-44s TC %.2e  FFMA2 %.2e  fp32 %.2e  gate %.2e" % row)
    table.append(row)


def kernels_ran(fn):
    """Names of the policy kernels a CUDA-activity profile of fn() shows."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return {k for k in TC | FFMA if any(k in n for n in names)}


def variant(R, v):
    return R._lib.load().rvb_policy_variant(v)


def net(R, sd, S, D, act, n_head, tanh, p=4):
    info = R.model.NetworkInfo([256, 160, 128], [80, 60], [80, 60], [80, 60], act)
    n = R.model._HeightmapNet(p + S + D, n_head, info, R.model.ObserverationInfo(p, S, D, 0), "cuda:0", tanh)
    n.load_state_dict(sd)
    return n


def run(R, a, obs, b=None, expect=TC):
    """One (b None) or a pair launch; asserts which kernels ran; returns the outputs."""
    out = []
    ran = kernels_ran(lambda: out.append(R.model.compute_pair(a, b, obs) if b is not None else (a._forward(obs),)))
    assert ran == expect, ran
    return out[0]


def ulp_diff(a, b):
    return ((a.view(torch.int32).long() - b.view(torch.int32).long()).abs().max()).item()


# ---------------------------------------------------------------------------------------------------------------- 1 + 2

@pytest.mark.parametrize("name", sorted(PP.probe_cases()))
def test_exact_probe(R, name):
    kw = PP.probe_cases()[name]
    pr = PP.make_exact_probe(**kw)
    other = PP.make_exact_probe(**dict(kw, obs=pr.obs, seed=kw["seed"] + 500))       # another network, same observations
    obs = pr.obs.cuda()
    a = net(R, pr.sd, pr.S, pr.D, pr.act, pr.n_head, pr.tanh)
    b = net(R, other.sd, pr.S, pr.D, pr.act, other.n_head, other.tanh)
    outs = {}
    try:
        for v, kernels in ((2, TC), (1, FFMA)):
            variant(R, v)
            single = run(R, a, obs, expect=kernels)[0].cpu()
            pa, pb = (t.cpu() for t in run(R, a, obs, b, expect=kernels))
            outs[v] = (single, pa, pb)
            for got, want in ((single, pr.expected), (pa, pr.expected), (pb, other.expected)):
                if pr.tanh:     # CUDA's tanhf is documented to 2 ulp (a 2-ulp case occurs in these probes on a B200)
                    assert ulp_diff(got, want) <= 2, (name, v)
                else:
                    assert torch.equal(got, want), (name, v, (got - want).abs().max().item())
    finally:
        variant(R, 2)
    # both paths feed the same exact fp32 sum into the same tanhf: the actor's outputs agree bit for bit as well
    for tc, ff in zip(outs[2], outs[1]):
        assert torch.equal(tc, ff), name


def _rand_sd(S, D, n_head, p, seed):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for name, (i, o) in {"es1": (S, 80), "es2": (80, 60), "ed1": (D, 80), "ed2": (80, 60), "m1": (p + 120, 256),
                         "m2": (256, 160), "m3": (160, 128), "head": (128, n_head)}.items():
        bd = 1 / i ** 0.5
        sd[PP.KEYS[name] + ".weight"] = (torch.rand(o, i, generator=g) * 2 - 1) * bd
        sd[PP.KEYS[name] + ".bias"] = (torch.rand(o, generator=g) * 2 - 1) * bd
    return sd


def _rand_obs(N, C, kind, seed, p=4):
    g = torch.Generator(device="cuda").manual_seed(seed)
    obs = torch.rand(N, C, device="cuda", generator=g) * 2 - 0.5
    half = (obs * 5.5 + 2.0).half().float()                          # heightmap-like: fp16 values in 0..8, no lo part
    if kind == "fp16":
        obs[:, p:] = half[:, p:]
    elif kind == "mixed":                                            # lo parts in some rows and some 32-column chunks only
        keep = (torch.rand(N, 1, device="cuda", generator=g) < 0.3) | \
               ((torch.arange(C, device="cuda") // 32) % 5 == 2)[None]
        obs[:, p:] = torch.where(keep[:, p:], obs[:, p:], half[:, p:])
    return obs


def _errors(R, a, obs, sd, p, S, D, act, tanh, b=None, sd_b=None, rows=None, expect=TC):
    """(TC error, FFMA2 error, torch fp32 error) against fp64, all on this device; max over the two networks of a pair."""
    ref_rows = obs if rows is None else obs[rows]
    errs = [0.0, 0.0, 0.0]
    nets = [(a, sd, tanh)] + ([(b, sd_b, False)] if b is not None else [])
    outs = {}
    for v in (2, 1):
        variant(R, v)
        outs[v] = run(R, a, obs, b, expect=expect if v == 2 else FFMA)
    variant(R, 2)
    for i, (_, s, t) in enumerate(nets):
        ref = PO.forward({k: x.cuda() for k, x in s.items()}, ref_rows, p, S, D, act, actor=t, dtype=torch.float64)
        f32 = PO.forward({k: x.cuda() for k, x in s.items()}, ref_rows, p, S, D, act, actor=t, dtype=torch.float32)
        for j, v in enumerate((2, 1)):
            o = outs[v][i] if rows is None else outs[v][i][rows]
            errs[j] = max(errs[j], PP.max_abs_err(o, ref))
        errs[2] = max(errs[2], PP.max_abs_err(f32, ref))
        del ref, f32
    return errs


# shapes: residues 26/24 (the shipped split), 0/2, 30/2, 2/0, 2/30 mod 32, and 65 chunks (> 64: the lo flags alias)
SWEEP = [
    # act,        S,    D,    N,    heads, tanh,  obs
    ("leakyrelu", 634, 1112, 4097, 2, True, "fp32"),
    ("leakyrelu", 634, 1112, 4097, 1, False, "fp16"),
    ("relu", 634, 1112, 383, 4, False, "mixed"),
    ("elu", 32, 2050, 129, 3, True, "fp32"),
    ("tanh", 62, 34, 128, 4, True, "mixed"),
    ("sigmoid", 2, 32, 127, 1, False, "fp32"),
    ("relu6", 2050, 62, 1, 2, False, "fp32"),
    ("relu", 34, 2050, 4097, 3, False, "mixed"),
    ("sigmoid", 1112, 634, 383, 2, True, "fp16"),
    ("elu", 634, 1112, 128, 1, False, "mixed"),
    ("tanh", 2050, 2050, 129, 4, False, "fp32"),
    ("relu6", 62, 32, 4097, 3, True, "mixed"),
]


@pytest.mark.parametrize("case", SWEEP, ids=lambda c: "%s-S%d-D%d-N%d-A%d-%s-%s" % (c[0], c[1], c[2], c[3], c[4],
                                                                                    "tanh" if c[5] else "lin", c[6]))
def test_dense_sweep_against_fp64(R, table, case):
    act, S, D, N, heads, tanh, kind = case
    sd = _rand_sd(S, D, heads, 4, seed=S * 7 + D + N)
    obs = _rand_obs(N, 4 + S + D, kind, seed=N + heads)
    a = net(R, sd, S, D, act, heads, tanh)
    tc, ff, f32 = _errors(R, a, obs, sd, 4, S, D, act, tanh)
    gate = PP.fp32_gate(f32)
    _record(table, ("-".join(map(str, case)), tc, ff, f32, gate))
    assert ff <= gate and tc <= gate, (tc, ff, f32)


@pytest.mark.parametrize("what", ["odd_ld", "offset_1", "odd_S", "odd_D", "p3", "p8", "variant1", "view_tc"])
def test_dispatch_and_fallbacks(R, table, what):
    """Which kernel serves which layout, and either path still meets the gate there."""
    S, D, p, expect = 634, 1112, 4, FFMA
    if what == "odd_S":
        S = 633
    elif what == "odd_D":
        D = 1111
    elif what in ("p3", "p8"):
        p = int(what[1])
    C = p + S + D
    wide = _rand_obs(300, C + 8, "fp32", seed=11)
    obs = wide[:, :C]
    if what == "odd_ld":
        obs = _rand_obs(300, C + 1, "fp32", seed=12)[:, :C]
    elif what == "offset_1":
        obs = wide[:, 1:C + 1]
    elif what == "view_tc":                    # strided, offset by 8 bytes: still the tensor-core path
        obs, expect = wide[:, 2:C + 2], TC
    sd = _rand_sd(S, D, 2, p, seed=3)
    a = net(R, sd, S, D, "leakyrelu", 2, True, p=p)
    if what == "variant1":
        variant(R, 1)
        try:
            ran = kernels_ran(lambda: a._forward(obs))
        finally:
            variant(R, 2)
        assert ran == FFMA
        return
    ran = kernels_ran(lambda: a._forward(obs))
    assert ran == expect, (what, ran)
    tc, ff, f32 = _errors(R, a, obs, sd, p, S, D, "leakyrelu", True, expect=expect)
    gate = PP.fp32_gate(f32)
    _record(table, ("dispatch-" + what, tc, ff, f32, gate))
    assert tc <= gate and ff <= gate, (tc, ff, f32)


# ---------------------------------------------------------------------------------------------------------------- 4

def test_step_observations_with_noise_pair(R, table):
    """The fused step's obs_buf, then ObsHooks' noise (arbitrary fp32: three-MMA chunks), actor + critic in one launch."""
    dev = "cuda:0"
    w = R.synth.make_world(length=12.0, nv=44, K=64, n_stones=8, seed=3, build_index=None)
    w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device=dev).cpu()
    kr = min(w.K, w.rock_triangles.shape[0])
    w.rock_indices = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, kr, device=dev).cpu()
    st = R.synth.make_env_state(w, 300, seed=5, margin=3.0)
    task = R.synth.make_task(w, st, device=dev, level=2)
    obs = task.hot_step(st["actions"].to(dev))[0].clone()
    assert obs.shape == (300, 1750)
    R.ObsHooks(1750, noise_std=math.sqrt(0.20)).apply(obs, epoch=1)
    assert bool((PP.split(obs[:, 4:])[1] != 0).any())
    sa, sc = _rand_sd(634, 1112, 2, 4, seed=41), _rand_sd(634, 1112, 1, 4, seed=42)
    a = net(R, sa, 634, 1112, "leakyrelu", 2, True)
    c = net(R, sc, 634, 1112, "leakyrelu", 1, False)
    tc, ff, f32 = _errors(R, a, obs, sa, 4, 634, 1112, "leakyrelu", True, b=c, sd_b=sc)
    gate = PP.fp32_gate(f32)
    _record(table, ("step+noise pair N=300", tc, ff, f32, gate))
    assert tc <= gate and ff <= gate, (tc, ff, f32)


def test_benchmark_size_pair_every_row(R, table):
    N = 131072
    sa, sc = _rand_sd(634, 1112, 2, 4, seed=51), _rand_sd(634, 1112, 1, 4, seed=52)
    a = net(R, sa, 634, 1112, "leakyrelu", 2, True)
    c = net(R, sc, 634, 1112, "leakyrelu", 1, False)
    obs = _rand_obs(N, 1750, "mixed", seed=53)
    tc, ff, f32 = _errors(R, a, obs, sa, 4, 634, 1112, "leakyrelu", True, b=c, sd_b=sc)
    gate = PP.fp32_gate(f32)
    _record(table, ("benchmark pair N=131072", tc, ff, f32, gate))
    assert tc <= gate and ff <= gate, (tc, ff, f32)


def test_observations_beyond_2_31_bytes_sampled(R, table):
    N = 320_000
    assert N * 1750 * 4 > 2 ** 31
    sa, sc = _rand_sd(634, 1112, 2, 4, seed=61), _rand_sd(634, 1112, 1, 4, seed=62)
    a = net(R, sa, 634, 1112, "leakyrelu", 2, True)
    c = net(R, sc, 634, 1112, "leakyrelu", 1, False)
    obs = _rand_obs(N, 1750, "fp32", seed=63)
    g = torch.Generator(device="cuda").manual_seed(64)
    rows = torch.cat((torch.randint(0, N, (4000,), device="cuda", generator=g), torch.arange(N - 200, N, device="cuda")))
    tc, ff, f32 = _errors(R, a, obs, sa, 4, 634, 1112, "leakyrelu", True, b=c, sd_b=sc, rows=rows)
    gate = PP.fp32_gate(f32)
    _record(table, ("pair N=320000 (sampled rows)", tc, ff, f32, gate))
    assert tc <= gate and ff <= gate, (tc, ff, f32)
