"""The policy and value networks on the step's packed observation (rvb_policy_forward_packed; model.compute / compute_pair on
(proprio f32, heightmap f16)).

The packed call must return the very bits of the f32 entry point on the widened rows cat(proprio, heightmap.float()), on the
tensor-core path and on the FFMA2 path, at every shape: through that identity it inherits every fp64-oracle check
tests/test_zz_gpu_policy_tc.py applies to the f32 path.  Every case names the kernels a torch.profiler trace shows; the
packed kernels have names of their own, and nothing else (no widening, no copy) runs.
"""
import pytest
import torch

import policy_oracle as PO
import policy_probe as PP

pytestmark = pytest.mark.gpu

TC16 = {"policy_l1_tc_h16_kernel", "policy_tail_tc_kernel"}
FFMA16 = {"policy_forward_h16_kernel"}
S0, D0 = 634, 1112


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


def kernels_ran(fn):
    """Names of every CUDA kernel / copy a CUDA-activity profile of fn() shows."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


def assert_ran(fn, expect):
    names = kernels_ran(fn)
    assert {k for k in expect if any(k in n for n in names)} == expect, names
    assert all(any(k in n for k in expect) for n in names), names            # nothing but the packed kernels


def variant(R, v):
    return R._lib.load().rvb_policy_variant(v)


def _rand_sd(S, D, n_head, p, seed):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for name, (i, o) in {"es1": (S, 80), "es2": (80, 60), "ed1": (D, 80), "ed2": (80, 60), "m1": (p + 120, 256),
                         "m2": (256, 160), "m3": (160, 128), "head": (128, n_head)}.items():
        bd = 1 / i ** 0.5
        sd[PP.KEYS[name] + ".weight"] = (torch.rand(o, i, generator=g) * 2 - 1) * bd
        sd[PP.KEYS[name] + ".bias"] = (torch.rand(o, generator=g) * 2 - 1) * bd
    return sd


def net(R, sd, S, D, n_head, tanh, p=4):
    info = R.model.NetworkInfo([256, 160, 128], [80, 60], [80, 60], [80, 60], "leakyrelu")
    n = R.model._HeightmapNet(p + S + D, n_head, info, R.model.ObserverationInfo(p, S, D, 0), "cuda:0", tanh)
    n.load_state_dict(sd)
    return n


def pair_nets(R, S=S0, D=D0, p=4, seed=0):
    sa, sc = _rand_sd(S, D, 2, p, seed + 1), _rand_sd(S, D, 1, p, seed + 2)
    return net(R, sa, S, D, 2, True, p), net(R, sc, S, D, 1, False, p), sa, sc


def packed_inputs(N, p, C, seed):
    """proprio f32 [N, p] and a heightmap f16 [N, C] like the ray-cast's (fp16(dist / 2), 0..8), with a few rows of extreme
    finite fp16 values: subnormals, -0, the largest finite value."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    proprio = torch.rand(N, p, device="cuda", generator=g) * 2 - 1
    hm = (torch.rand(N, C, device="cuda", generator=g) * 8).half()
    if N > 8:
        hm[1, ::3] = torch.tensor(2.0 ** -24, dtype=torch.float16)
        hm[2, ::5] = torch.tensor(-0.0, dtype=torch.float16)
        hm[3, ::7] = torch.tensor(65504.0, dtype=torch.float16)
        hm[4] = -hm[4]
    return proprio, hm


def widened(proprio, hm):
    return torch.cat((proprio, hm.float()), 1)


def compare(R, a, b, proprio, hm, expect, ref_variant=None):
    """The packed call (one network, and the pair when b is given) against the f32 entry point on the widened rows, under the
    current dispatch (or ref_variant for the f32 reference); asserts the kernels and returns the outputs."""
    ref_states = widened(proprio, hm)
    prev = variant(R, ref_variant) if ref_variant else None
    try:
        ref1 = a._forward(ref_states)
        refp = R.model.compute_pair(a, b, ref_states) if b is not None else None
    finally:
        if prev:
            variant(R, prev)
    got = []
    assert_ran(lambda: got.append(a._forward((proprio, hm))), expect)
    assert torch.equal(got[0], ref1)
    if b is not None:
        assert_ran(lambda: got.append(R.model.compute_pair(a, b, (proprio, hm))), expect)
        assert torch.equal(got[1][0], refp[0]) and torch.equal(got[1][1], refp[1])
        assert torch.equal(got[1][0], got[0])                                 # one network = its half of the pair
    return got


# ---------------------------------------------------------------------------------------------------------------- 1

@pytest.mark.parametrize("N", [1, 127, 128, 129, 4097, 131072])
@pytest.mark.parametrize("v", [2, 1])
def test_bit_identity_shipped_shape(R, N, v):
    a, c, _, _ = pair_nets(R, seed=10)
    proprio, hm = packed_inputs(N, 4, S0 + D0, seed=N)
    prev = variant(R, v)
    try:
        compare(R, a, c, proprio, hm, TC16 if v == 2 else FFMA16)
    finally:
        variant(R, prev)


@pytest.mark.parametrize("v", [2, 1])
def test_non_finite_heightmap_values(R, v):
    """+-inf and NaN in the fp16 heightmap: the rows that hold them come out as the f32 entry point makes them (NaN on the
    tensor-core path, where the f32 split's lo part of an infinity is NaN), every other row bit for bit."""
    a, c, _, _ = pair_nets(R, seed=20)
    proprio, hm = packed_inputs(300, 4, S0 + D0, seed=21)
    hm[5, 7] = float("inf")
    hm[6, S0 + 3] = -float("inf")
    hm[7, 100] = float("nan")
    prev = variant(R, v)
    try:
        ref = R.model.compute_pair(a, c, widened(proprio, hm))
        got = R.model.compute_pair(a, c, (proprio, hm))
    finally:
        variant(R, prev)
    for x, y in zip(got, ref):
        torch.testing.assert_close(x, y, rtol=0, atol=0, equal_nan=True)
        assert bool(torch.isnan(y[7]).all())


# ---------------------------------------------------------------------------------------------------------------- 2

@pytest.mark.parametrize("what", ["odd_ld", "offset_1", "offset_2", "odd_S", "odd_D", "p3", "p8", "proprio_view"])
def test_fallbacks(R, what):
    """Each layout the tensor-core path refuses runs the FFMA2 kernel, bit for bit what the f32 entry point returns on the same
    path; a heightmap offset by two halves (4-byte aligned) and the strided view obs_buf[:, :4] stay on the tensor cores."""
    S, D, p, expect = S0, D0, 4, FFMA16
    if what == "odd_S":
        S = 633
    elif what == "odd_D":
        D = 1111
    elif what in ("p3", "p8"):
        p = int(what[1])
    N, C = 300, S + D
    proprio, wide = packed_inputs(N, p, C + 8, seed=31)
    hm = wide[:, :C]
    if what == "odd_ld":
        hm = packed_inputs(N, p, C + 1, seed=32)[1][:, :C]
    elif what == "offset_1":
        hm = wide[:, 1:C + 1]
    elif what == "offset_2":
        hm, expect = wide[:, 2:C + 2], TC16
    elif what == "proprio_view":
        obs_buf = torch.rand(N, p + C, device="cuda")
        proprio, expect = obs_buf[:, :p], TC16
        assert proprio.stride(0) == p + C
    a, c, _, _ = pair_nets(R, S, D, p, seed=33)
    compare(R, a, c, proprio, hm, expect, ref_variant=2 if expect == TC16 else 1)


def test_short_rows_and_mismatched_networks_are_refused(R):
    lib = R._lib.load()
    ptr = R._lib.ptr
    a, c, _, _ = pair_nets(R, seed=40)
    proprio, hm = packed_inputs(130, 4, S0 + D0, seed=41)
    out = torch.empty(130, 2, device="cuda")

    def call(b, proprio_ld, hm_ld, out_ld):
        return lib.rvb_policy_forward_packed(a._handle, b._handle if b is not None else None, ptr(proprio), proprio_ld, ptr(hm), hm_ld,
                                             130, ptr(out), out_ld, ptr(out), 2, None)
    assert call(None, 3, S0 + D0, 2) == -1 and b"proprio rows are shorter" in lib.rvb_last_error()
    assert call(None, 4, S0 + D0 - 1, 2) == -1 and b"heightmap rows are shorter" in lib.rvb_last_error()
    assert call(None, 4, S0 + D0, 1) == -1 and b"out rows are shorter" in lib.rvb_last_error()
    relu = R.model._HeightmapNet(1750, 1, R.model.NetworkInfo([256, 160, 128], [80, 60], [80, 60], [80, 60], "relu"),
                                 R.model.ObserverationInfo(4, S0, D0, 0), "cuda:0", False)
    assert call(relu, 4, S0 + D0, 2) == -1 and b"different activations" in lib.rvb_last_error()
    assert call(c, 4, S0 + D0, 2) == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------- 3

@pytest.fixture(scope="module")
def world(R):
    dev = "cuda:0"
    w = R.synth.make_world(length=12.0, nv=44, K=64, n_stones=8, seed=3, build_index=None)
    w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device=dev).cpu()
    kr = min(w.K, w.rock_triangles.shape[0])
    w.rock_indices = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, kr, device=dev).cpu()
    return w


def test_step_feeds_the_networks(R, world):
    """RoverTask.hot_step with and without obs16_buf, from the same poses and actions (curriculum level 2, the second step with
    the device-side reset): compute_pair on (obs_buf[:, :4], obs16_buf) equals compute_pair on the f32 obs_buf bit for bit."""
    dev = "cuda:0"
    N = 300
    st = R.synth.make_env_state(world, N, seed=5, margin=3.0)
    t32 = R.synth.make_task(world, st, device=dev, level=2)
    t16 = R.synth.make_task(world, st, device=dev, level=2)
    t16.obs16_buf = torch.zeros((N, 1746), dtype=torch.float16, device=dev)
    a, c, _, _ = pair_nets(R, seed=50)
    for k in range(2):
        act = (st["actions"] * (1.0 - 0.25 * k)).to(dev)
        obs = t32.hot_step(act, device_reset=(k == 1))[0]
        t16.hot_step(act, device_reset=(k == 1))
        assert torch.equal(t16.obs16_buf.float(), obs[:, 4:]) and torch.equal(t16.obs_buf[:, :4], obs[:, :4])
        ref = R.model.compute_pair(a, c, obs)
        got = []
        assert_ran(lambda: got.append(R.model.compute_pair(a, c, (t16.obs_buf[:, :4], t16.obs16_buf))), TC16)
        assert torch.equal(got[0][0], ref[0]) and torch.equal(got[0][1], ref[1])


def test_host_pipeline_packed_slots_feed_the_networks(R, world):
    """HostPipeline(packed_obs=True, device_reset=True): the slot's device buffers feed compute_pair as they are."""
    N = 200
    st = R.synth.make_env_state(world, N, seed=33, margin=3.0)
    p32 = R.HostPipeline(R.synth.make_task(world, st, device="cuda:0", level=2), device_reset=True)
    p16 = R.HostPipeline(R.synth.make_task(world, st, device="cuda:0", level=2), packed_obs=True, device_reset=True)
    a, c, _, _ = pair_nets(R, seed=60)
    g = torch.Generator().manual_seed(2)
    hs = {k: v.clone() for k, v in st.items()}
    for step in range(3):
        act = torch.rand(N, 2, generator=g) * 2 - 1
        hs["pos"][:, 1] += 0.02
        k32 = p32.submit(hs["pos"], hs["quat"], hs["joints"], act)
        k16 = p16.submit(hs["pos"], hs["quat"], hs["joints"], act)
        p32.result(k32)
        p16.result(k16)
        ref = R.model.compute_pair(a, c, p32.d_obs[k32])
        got = R.model.compute_pair(a, c, (p16.d_obs[k16][:, :4], p16.d_obs16[k16]))
        assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1]), step
    p32.close()
    p16.close()


# ---------------------------------------------------------------------------------------------------------------- 4

def test_heightmap_beyond_2_31_bytes(R):
    N = 620_000
    assert N * (S0 + D0) * 2 > 2 ** 31
    a, c, sa, sc = pair_nets(R, seed=70)
    proprio, hm = packed_inputs(N, 4, S0 + D0, seed=71)
    got = R.model.compute_pair(a, c, (proprio, hm))
    obs = widened(proprio, hm)
    ref = R.model.compute_pair(a, c, obs)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    g = torch.Generator(device="cuda").manual_seed(72)
    rows = torch.cat((torch.randint(0, N, (4000,), device="cuda", generator=g), torch.arange(N - 200, N, device="cuda")))
    sub = obs[rows]
    del obs, ref
    for out, sd, actor in ((got[0], sa, True), (got[1], sc, False)):
        sdc = {k: x.cuda() for k, x in sd.items()}
        ref64 = PO.forward(sdc, sub, 4, S0, D0, "leakyrelu", actor=actor, dtype=torch.float64)
        f32 = PO.forward(sdc, sub, 4, S0, D0, "leakyrelu", actor=actor, dtype=torch.float32)
        err, err32 = PP.max_abs_err(out[rows], ref64), PP.max_abs_err(f32, ref64)
        print("packed pair N=620000 (sampled rows) %s: err %.2e  fp32 %.2e  gate %.2e" % ("actor" if actor else "critic", err, err32,
                                                                                         PP.fp32_gate(err32)))
        assert err <= PP.fp32_gate(err32), (err, err32)
