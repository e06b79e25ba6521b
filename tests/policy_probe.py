"""Helpers for the policy network's tensor-core path (csrc/policy.cu, policy_l1_tc_kernel + policy_tail_tc_kernel).

emulate_tc(): the arithmetic of that path in torch -- every operand of the seven tcgen05 layers split into tf32 hi + lo
(cvt.rna.tf32.f32), the products Ah.Wh + Ah.Wl + Al.Wh summed in fp32, bias and activation in fp32, the head an fp32 FMA
chain -- with the mutations a subtly wrong kernel would show (a missing lo MMA, single-pass tf32, two swapped features,
a skipped tile row), and two models of the accumulator: exact sum + one rounding ("rn"), or a round-toward-zero after every
MMA of eight products ("rz", the truncating alignment the tensor cores of earlier generations are documented to use).

make_exact_probe(): networks and observations on which fp32 arithmetic in ANY summation order, with any accumulator
rounding, is exact, so a correct kernel returns the fp64 oracle's answer bit for bit (the actor: up to the 2 ulp of
CUDA's tanhf).
The generator checks its own invariants in fp64 (every value below is an integer multiple of a power of two well inside
fp64's 53 bits, so those checks are exact) and raises if one fails:
  1. every weight and bias has <= 11 significant bits (tf32 lo part 0: the Al.Wl term the kernel omits is 0);
  2. every value fed into a tensor-core layer has <= 22 significant bits (hi + lo == x exactly);
  3. per layer, every term x_k * w_jk and bias b_j is a multiple of the layer's quantum q, and sum |terms| + |b| < 2^24 q,
     so every partial sum in every order is an fp32 number;
  4. every activation fed on is < 2^22 q;
  5. only exact activations: relu, relu6, and leakyrelu with positive pre-activations;
  6. the critic head has no tanh (the actor's answer depends on the tanh implementation by a few ulp).
Construction: first layers +-2^-5 with random signs on observations m * 2^-14 (m of 12-13 bits: about half carry a lo
part) or on "coarse" values k * 2^-8 (|k| < 16: no lo part); every later layer is a fan-in-one routing with weight 1 and a
positive bias k * 2^-8, so a value keeps its bits from the first layer to the head; the head sums up to four routed paths
with weights +-1 or +-1/2.  A path runs from one concat feature (proprio column, sparse or dense encoder output) through
chosen features of the 256-, 160- and 128-wide layers to one head output.
"""
import torch

import policy_oracle

P = 4                         # proprio columns on the tensor-core path (tc_usable)
E1, E2, M1, M2, M3 = 80, 60, 256, 160, 128
LAYERS = ("es1", "ed1", "es2", "ed2", "m1", "m2", "m3")
KEYS = {"es1": "encoder0.encoder.0.layer.0", "es2": "encoder0.encoder.1.layer.0", "ed1": "encoder1.encoder.0.layer.0",
        "ed2": "encoder1.encoder.1.layer.0", "m1": "network.0.layer.0", "m2": "network.1.layer.0", "m3": "network.2.layer.0",
        "head": "network.3"}
EXACT_ACTS = ("relu", "relu6", "leakyrelu")


def tf32(x):
    """cvt.rna.tf32.f32: round to nearest, ties away from zero, to 10 explicit mantissa bits (result kept as f32)."""
    b = x.to(torch.float32).contiguous().view(torch.int32).to(torch.int64)
    b = (b + 0x1000) & ~0x1FFF
    return b.to(torch.int32).view(torch.float32)


def split(x):
    """x -> (hi, lo) as the kernels split it: hi = tf32(x), lo = tf32(x - hi) (the difference is exact in fp32)."""
    hi = tf32(x)
    return hi, tf32(x.to(torch.float32) - hi)


def _act(v, act):
    return policy_oracle.ACTIVATIONS[act](v)


def _round_rz(v):
    """fp64 -> the fp32 value next to it toward zero."""
    f = v.to(torch.float32)
    over = f.double().abs() > v.abs()
    return torch.where(over, torch.nextafter(f, torch.zeros_like(f)), f)


def _tc_linear(x, w, b, act, drop_lo=None, single=False, acc="rn"):
    """act(x . w^T + b) as one tensor-core layer computes it.  x f32 [N, K], w f32 [O, K], b f32 [O].
    drop_lo: None, "all", or a chunk index c: the Al.Wh MMA of those 32-column chunks is not issued."""
    xh, xl = split(x)
    wh, wl = split(w)
    if single:
        xl = torch.zeros_like(xl)
        wl = torch.zeros_like(wl)
    if drop_lo == "all":
        xl = torch.zeros_like(xl)
    elif drop_lo is not None:
        xl = xl.clone()
        xl[:, 32 * drop_lo:32 * drop_lo + 32] = 0
    xh, xl, wh, wl = (t.double() for t in (xh, xl, wh, wl))
    if acc == "rn":                                    # products are exact (22 bits); fp64 sums them with negligible error
        y = (xh @ wh.T + xh @ wl.T + xl @ wh.T).to(torch.float32)
    else:                                              # "rz": truncate after every MMA of 8 products (order Ah.Wh, Ah.Wl, Al.Wh)
        y = torch.zeros(x.shape[0], w.shape[0], dtype=torch.float32)
        for k0 in range(0, x.shape[1], 8):
            s = slice(k0, k0 + 8)
            for a, bb in ((xh, wh), (xh, wl), (xl, wh)):
                y = _round_rz(y.double() + a[:, s] @ bb[:, s].T)
    return _act(y + b.to(torch.float32), act)


def emulate_tc(sd, obs, S, D, act="leakyrelu", tanh=False, drop_lo=None, single=False, swap=None, skip_row=None, acc="rn"):
    """The tensor-core path's answer for state dict `sd` (reference keys) on f32 observations [N, >= 4 + S + D].
    drop_lo:  None | "all" (both first layers) | ("s" | "d", c): the lo MMA of first-layer chunk c is never issued;
    single:   single-pass tf32 in every tensor-core layer (no lo parts at all);
    swap:     (layer, f): that layer reads input features f - 1 and f swapped (layer in LAYERS; es1 / ed1 count columns from
              the start of the encoder's slice);
    skip_row: r: the first layers read row r of every 128-row tile as zeros;
    acc:      "rn" (exact accumulation, one rounding) or "rz" (see _tc_linear).
    Returns f32 [N, A]."""
    W = {n: sd[KEYS[n] + ".weight"].to(torch.float32) for n in KEYS}
    B = {n: sd[KEYS[n] + ".bias"].to(torch.float32) for n in KEYS}
    obs = obs.to(torch.float32)
    if skip_row is not None:
        obs = obs.clone()
        obs[skip_row::128] = 0

    def lin(name, x, **kw):
        if swap is not None and swap[0] == name:
            f = swap[1]
            x = x.clone()
            x[:, [f - 1, f]] = x[:, [f, f - 1]]
        return _tc_linear(x, W[name], B[name], act, single=single, acc=acc, **kw)

    def first(enc):
        if drop_lo == "all":
            return "all"
        if drop_lo is not None and drop_lo[0] == enc:
            return drop_lo[1]
        return None
    xs = obs[:, P:P + S]
    xd = obs[:, P + S:P + S + D]
    x0 = lin("es2", lin("es1", xs, drop_lo=first("s")))
    x1 = lin("ed2", lin("ed1", xd, drop_lo=first("d")))
    h = torch.cat((obs[:, :P], x0, x1), 1)
    h = lin("m3", lin("m2", lin("m1", h)))
    y = (h.double() @ W["head"].double().T).to(torch.float32) + B["head"]
    return torch.tanh(y.double()).to(torch.float32) if tanh else y


# ------------------------------------------------------------------------------------------------------------------
# exact probes

class Probe:
    """sd: state dict (reference keys, f32); obs: f32 [N, 4 + S + D]; expected: f32 [N, A], the fp64 oracle's answer
    (exactly an fp32 number before the actor's tanh); pre: the head's fp64 output before tanh; paths: the routed paths."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def probe_obs(N, S, D, fine=None, seed=0):
    """Observations: `fine` is a list of (rows, cols) index pairs (cols absolute, >= 4) whose entries get m * 2^-14 with an
    odd m of 12-13 significant bits (so every one has a lo part) and a random sign; every other exteroceptive entry gets a
    coarse k * 2^-8, |k| < 16 (no lo part).  fine=None makes every exteroceptive entry fine, m of any parity (about half
    have a lo part).  Proprio columns: positive m * 2^-14 in every row."""
    g = torch.Generator().manual_seed(seed)
    C = P + S + D

    def finevals(shape, odd=False):
        m = torch.randint(1 << 11, 1 << 13, shape, generator=g, dtype=torch.int64) | int(odd)
        s = torch.randint(0, 2, shape, generator=g) * 2 - 1
        return (m * s).double() * 2.0 ** -14
    obs = torch.randint(-15, 16, (N, C), generator=g).double() * 2.0 ** -8
    if fine is None:
        obs[:, P:] = finevals((N, C - P))
    else:
        for rows, cols in fine:
            r = torch.as_tensor(rows).reshape(-1, 1)
            c = torch.as_tensor(cols).reshape(1, -1)
            obs[r, c] = finevals((r.shape[0], c.shape[1]), odd=True)
    obs[:, :P] = finevals((N, P)).abs()               # positive: a routed proprio column stays positive for leakyrelu
    return obs.to(torch.float32)


def _route(n_head, seed, concat=None, m1=None, m2=None, m3=None):
    """Paths (concat feature, m1 feature, m2 feature, m3 feature, head output): four per head output (at most 16).
    Defaults put paths on chunk-boundary features of every tensor-core input, on both halves of the 256-wide layer, on
    features 128-159 of the 160-wide layer, and on every proprio column."""
    g = torch.Generator().manual_seed(seed)
    n = 4 * n_head

    def perm(k, first=(), base=0):
        """first, then the other features of [base, base + k) in random order"""
        return list(first) + [base + i for i in torch.randperm(k, generator=g).tolist() if base + i not in first]
    if concat is None:
        pool = [0, 1, 2, 3, 31, 32, 63, 64, 95, 96, 123, 4, 35, 67, 100, 127 - 4]
        concat = [pool[i] for i in perm(len(pool))][:n]
    if m1 is None:                                     # alternate halves: the second half is the second TMEM pass (D3 + 128)
        lo, hi = perm(128, (127,)), perm(128, (128,), 128)
        m1 = [(hi if i % 2 else lo)[i // 2] for i in range(n)]
    if m2 is None:                                     # features 128-159: the second pass of the 160-wide layer
        lo, hi = perm(128, (127,)), perm(32, (128,), 128)
        m2 = [(hi if i % 2 else lo)[i // 2] for i in range(n)]
    if m3 is None:
        m3 = perm(M3, (31, 32))[:n]
    return [(concat[i], m1[i], m2[i], m3[i], i % n_head) for i in range(n)]


def _routing_layer(n_out, n_in, pairs, gen, bias_k=64):
    """Fan-in-one weights: out feature j <- in feature src[j] with weight 1; positive biases k * 2^-8."""
    w = torch.zeros(n_out, n_in, dtype=torch.float64)
    for j, i in pairs:
        w[j, i] = 1.0
    b = torch.randint(1, bias_k, (n_out,), generator=gen).double() * 2.0 ** -8
    return w, b


def _check_layer(name, x, w, b, q, act):
    """Invariants 1-5 on one layer in fp64: x [N, K] (exact values), w [O, K], b [O]; returns the activation."""
    for t, what in ((w, "weight"), (b, "bias")):
        assert torch.equal(tf32(t).double(), t), "%s %s: more than 11 significant bits" % (name, what)          # 1
    hi = tf32(x).double()
    lo = tf32((x - hi)).double()
    assert torch.equal(hi + lo, x), "%s input: more than 22 significant bits" % name                          # 2
    assert bool(((x / q).abs() < 2.0 ** 22).all()), "%s input: not below 2^22 q" % name                       # 4
    for t, what in ((x[:, None, :] * w[None], "terms"), (b, "bias")):
        u = t / q
        assert torch.equal(u, u.round()), "%s %s: not multiples of the quantum" % (name, what)               # 3
    big = (x.abs() @ w.abs().T + b.abs()) / q
    assert bool((big < 2.0 ** 24).all()), "%s: sum |terms| + |b| >= 2^24 q" % name                            # 3
    pre = x @ w.T + b
    if act == "leakyrelu":
        assert bool((pre > 0).all()), "%s: leakyrelu needs positive pre-activations" % name                   # 5
    return policy_oracle.ACTIVATIONS[act](pre)


def make_exact_probe(S=634, D=1112, n_head=4, act="relu", tanh=False, N=130, fine=None, obs=None, seed=0, paths=None,
                     **route):
    """A network (and observations, unless `obs` is given) on which the tensor-core path must return the fp64 oracle's
    answer bit for bit.  See the module docstring for the construction; raises AssertionError if an invariant fails."""
    assert act in EXACT_ACTS, "only exact activations: %s" % (EXACT_ACTS,)                                  # 5
    assert 1 <= n_head <= 4
    g = torch.Generator().manual_seed(1000 + seed)
    if obs is None:
        obs = probe_obs(N, S, D, fine, seed)
    N = obs.shape[0]
    x = obs.double()
    q1 = 2.0 ** -19                                    # observation quantum 2^-14 x first-layer weight 2^-5
    paths = paths or _route(n_head, seed, **route)
    sd = {}

    def put(name, w, b):
        sd[KEYS[name] + ".weight"] = w.to(torch.float32)
        sd[KEYS[name] + ".bias"] = b.to(torch.float32)
    # first layers: +-2^-5, biases that make every pre-activation positive (a positive multiple of q1)
    acts = {}
    for name, cols in (("es1", slice(P, P + S)), ("ed1", slice(P + S, P + S + D))):
        K = cols.stop - cols.start
        w = (torch.randint(0, 2, (E1, K), generator=g).double() * 2 - 1) * 2.0 ** -5
        s = x[:, cols] @ w.T
        need = (-s.min(0).values).clamp(min=0)         # bias k * 2^-8 (<= 11 bits below 8) above every negative sum
        b = (torch.floor(need * 2.0 ** 8) + torch.randint(1, 16, (E1,), generator=g).double()) * 2.0 ** -8
        put(name, w, b)
        acts[name] = _check_layer(name, x[:, cols], w, b, q1, act)
    # second encoder layers: every output routes one first-layer feature
    for name, src in (("es2", "es1"), ("ed2", "ed1")):
        w, b = _routing_layer(E2, E1, [(j, int(i)) for j, i in enumerate(torch.randperm(E1, generator=g)[:E2])], g)
        put(name, w, b)
        acts[name] = _check_layer(name, acts[src], w, b, q1, act)
    h = torch.cat((x[:, :P], acts["es2"], acts["ed2"]), 1)
    chain = (("m1", 2 * E2 + P, M1, 1), ("m2", M1, M2, 2), ("m3", M2, M3, 3))
    for name, n_in, n_out, slot in chain:
        src = {}
        for pth in paths:
            prev = pth[slot - 1]
            assert src.get(pth[slot], prev) == prev, "two paths want feature %d of %s from different inputs" % (pth[slot], name)
            src[pth[slot]] = prev
        w, b = _routing_layer(n_out, n_in, sorted(src.items()), g)
        put(name, w, b)
        h = _check_layer(name, h, w, b, q1, act)
    # head: up to four paths per output, weights +-1 or +-1/2, bias +-k * 2^-8
    wh = torch.zeros(n_head, M3, dtype=torch.float64)
    for pth in paths:
        sign = torch.randint(0, 2, (1,), generator=g).item() * 2 - 1
        wh[pth[4], pth[3]] = sign * 2.0 ** -torch.randint(0, 2, (1,), generator=g).item()
    bh = (torch.randint(-63, 64, (n_head,), generator=g).double()) * 2.0 ** -8
    sd[KEYS["head"] + ".weight"] = wh.to(torch.float32)
    sd[KEYS["head"] + ".bias"] = bh.to(torch.float32)
    pre = h @ wh.T + bh
    qh = q1 / 2                                        # head weights +-1/2 halve the quantum
    big = (h.abs() @ wh.abs().T + bh.abs()) / qh
    assert bool((big < 2.0 ** 24).all()) and torch.equal(pre / qh, (pre / qh).round()), "head sum is not exact in fp32"
    assert torch.equal(pre.to(torch.float32).double(), pre)
    # the construction and the repository's fp64 oracle agree exactly
    ref = policy_oracle.forward(sd, obs, P, S, D, act, actor=tanh, dtype=torch.float64)
    assert torch.equal(ref, torch.tanh(pre) if tanh else pre), "fp64 oracle differs from the probe's own forward pass"
    return Probe(sd=sd, obs=obs, expected=ref.to(torch.float32), pre=pre, paths=paths, S=S, D=D, act=act, tanh=tanh,
                 n_head=n_head)


def probe_cases():
    """The named exact probes (name -> kwargs of make_exact_probe), the set the CPU and GPU tests share."""
    S, D = 634, 1112
    sp, dn = P, P + S                                  # first column of the sparse / dense slice
    cases = {
        "dense_all_fine": dict(S=S, D=D, n_head=4, act="relu", N=300, seed=1),
        "dense_leaky_head2": dict(S=S, D=D, n_head=2, act="leakyrelu", N=130, seed=2),
        "relu6_head3_tanh": dict(S=S, D=D, n_head=3, act="relu6", tanh=True, N=129, seed=3),
        "head1": dict(S=S, D=D, n_head=1, act="relu", N=1, seed=4),
        "aliased_chunks": dict(S=62, D=2050, n_head=4, act="leakyrelu", N=200, seed=5),
    }
    # lo parts in one chunk of one row only: rows 0, 127 and the last live row of a ragged tile (N = 130: row 129)
    for row in (0, 127, 129):
        for enc, c0, last in (("s", sp, S), ("d", dn, D)):
            cases["lo_row%d_%s_chunk0" % (row, enc)] = dict(S=S, D=D, N=130, seed=10 + row, fine=[([row], range(c0, c0 + 32))])
            c = (last - 1) // 32                       # the last, partial chunk: its last two columns
            cases["lo_row%d_%s_last" % (row, enc)] = dict(S=S, D=D, N=130, seed=20 + row,
                                                         fine=[([row], range(c0 + last - 2, c0 + last))])
    # chunk 64 of a 65-chunk encoder (its lo flag shares a slot with chunk 0)
    cases["lo_chunk64_only"] = dict(S=62, D=2050, N=130, seed=30, fine=[([5], range(P + 62 + 2048, P + 62 + 2050))])
    return cases


def max_abs_err(got, ref):
    """max |got - ref| (fp64), the error measure of the statistical gate."""
    return (got.double() - ref.double()).abs().max().item()


def fp32_gate(err_fp32):
    """The dense sweep's gate: the tensor-core path must stay within 32x of what torch fp32 makes of the same case."""
    return max(32.0 * err_fp32, 1e-7)
