"""Policy / value inference on obs_buf -- mirror of the reference's learning/model.py (SURVEY.md 8f-3).

Same class names, constructor arguments and `compute()` results as `StochasticActorHeightmap` (model.py:152-195) and
`DeterministicHeightmap` (model.py:197-241); parameters are exchanged through `state_dict()` / `load_state_dict()` with
the reference's key names (`encoder0.encoder.0.layer.0.weight`, ..., `network.3.weight`, `log_std_parameter`), so a
checkpoint of the reference's nn.Modules loads as is.  The forward pass is ONE kernel behind the C ABI
(`rvb_policy_forward`, csrc/policy.cu); skrl's mixins (sampling, clipping, log-prob) are the learner's and stay outside.
`states` is the f32 observation [N, >=p+S+D] or, from a step run in packed mode, the 2-tuple (proprio f32 [N, >=p],
heightmap f16 [N, >=S+D]), e.g. `(task.obs_buf[:, :4], task.obs16_buf)`: same results bit for bit as on the widened rows, read
without widening (`rvb_policy_forward_packed`).
Inference only: there is no autograd through the kernel.
"""
import ctypes as C
import math

import torch

from . import _lib


class ObserverationInfo:
    """model.py:10-41 (spelling as in the reference)."""

    def __init__(self, num_proprioceptive, num_sparse, num_dense, num_beneath):
        self.num_proprioceptive = num_proprioceptive
        self.num_sparse = num_sparse
        self.num_dense = num_dense
        self.num_beneath = num_beneath

    def get_num_proprioceptive(self):
        return self.num_proprioceptive

    def get_num_sparse(self):
        return self.num_sparse

    def get_num_dense(self):
        return self.num_dense

    def get_num_beneath(self):
        return self.num_beneath


class NetworkInfo:
    """model.py:43-66."""

    def __init__(self, network_0, encoder_0, encoder_1, encoder_2, activation_function):
        self.mlp_features = network_0
        self.sparse_encoder_features = encoder_0
        self.dense_encoder_features = encoder_1
        self.beneath_encoder_features = encoder_2
        self.activation_function = activation_function

    def get_mlp_features(self):
        return self.mlp_features

    def get_sparse_encoder_features(self):
        return self.sparse_encoder_features

    def get_dense_encoder_features(self):
        return self.dense_encoder_features

    def get_beneath_encoder_features(self):
        return self.beneath_encoder_features

    def get_activation_function(self):
        return self.activation_function


def _space_dim(space):
    if isinstance(space, int):
        return space
    return int(space.shape[0])


def _linear_keys(prefix):
    return prefix + ".weight", prefix + ".bias"


class _HeightmapNet:
    """Shared body of the two reference models: encoders + MLP + a final nn.Linear (model.py:162-177, 214-229)."""

    def __init__(self, observation_space, head_out, networkInfo, observartionInfo, device, head_tanh):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("rover_b200: the policy needs a CUDA device (there is no CPU path)")
        self.num_sparse = observartionInfo.get_num_sparse()
        self.num_dense = observartionInfo.get_num_dense()
        self.num_beneath = observartionInfo.get_num_beneath()
        self.mlp_features = list(networkInfo.get_mlp_features())
        self.sparse_features = list(networkInfo.get_sparse_encoder_features())
        self.dense_features = list(networkInfo.get_dense_encoder_features())
        self.beneath_features = networkInfo.get_beneath_encoder_features()
        self.activation_function = networkInfo.get_activation_function()
        if self.activation_function not in _lib.ACTIVATIONS:
            raise KeyError(self.activation_function)                     # like the dict lookup of model.py:114
        self.num_exteroceptive = self.num_sparse + self.num_dense
        self.num_observations = _space_dim(observation_space)
        self.num_proprioception = self.num_observations - self.num_exteroceptive     # model.py:167 overrides the info's value
        self._head_out = head_out
        self._head_tanh = head_tanh
        self._handle = None
        self._lib = _lib.load()
        # parameter table in the reference's module order, nn.Linear default initialisation
        self._layout = []
        for enc, n_in, feats in (("encoder0", self.num_sparse, self.sparse_features), ("encoder1", self.num_dense, self.dense_features)):
            c = n_in
            for i, f in enumerate(feats):
                self._layout.append(("%s.encoder.%d.layer.0" % (enc, i), c, f))
                c = f
        c = self.num_proprioception + self.dense_features[-1] + self.sparse_features[-1]
        for i, f in enumerate(self.mlp_features):
            self._layout.append(("network.%d.layer.0" % i, c, f))
            c = f
        self._layout.append(("network.%d" % len(self.mlp_features), c, head_out))
        self._params = {}
        for name, n_in, n_out in self._layout:
            bound = 1.0 / math.sqrt(n_in)
            wk, bk = _linear_keys(name)
            self._params[wk] = (torch.rand(n_out, n_in) * 2 - 1) * bound
            self._params[bk] = (torch.rand(n_out) * 2 - 1) * bound
        self._rebuild()

    # ---- parameters
    def _extra_state(self):
        return {}

    def state_dict(self):
        d = {k: v.clone() for k, v in self._params.items()}
        d.update(self._extra_state())
        return d

    def load_state_dict(self, sd, strict=True):
        for name, n_in, n_out in self._layout:
            for key, shape in zip(_linear_keys(name), ((n_out, n_in), (n_out,))):
                if key not in sd:
                    if strict:
                        raise KeyError(key)
                    continue
                t = torch.as_tensor(sd[key]).detach().to("cpu", torch.float32)
                if tuple(t.shape) != shape:
                    raise RuntimeError("size mismatch for %s: %s vs %s" % (key, tuple(t.shape), shape))
                self._params[key] = t.clone()
        self._load_extra(sd)
        self._rebuild()

    def _load_extra(self, sd):
        pass

    def _rebuild(self):
        self.close()
        dev = {k: v.to(self.device, torch.float32).contiguous() for k, v in self._params.items()}

        def arr(names):
            a = (_lib.Linear * len(names))()
            for i, n in enumerate(names):
                w, b = dev[n + ".weight"], dev[n + ".bias"]
                a[i] = _lib.Linear(w.data_ptr(), b.data_ptr(), w.shape[1], w.shape[0])
            return a
        names = [n for n, _, _ in self._layout]
        ns, nd, nm = len(self.sparse_features), len(self.dense_features), len(self.mlp_features)
        if (ns, nd, nm) != (2, 2, 3):
            raise RuntimeError("rover_b200: the policy kernel implements the reference network (2-layer encoders, 3-layer mlp; "
                               "train.py:95)")
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            _lib.check(self._lib.rvb_policy_create(C.byref(h), self.num_proprioception, self.num_sparse, self.num_dense,
                                                   arr(names[0:ns]), arr(names[ns:ns + nd]), arr(names[ns + nd:ns + nd + nm]),
                                                   arr(names[-1:]), _lib.ACTIVATIONS[self.activation_function],
                                                   1 if self._head_tanh else 0, torch.cuda.current_device(), st))
        self._handle = h

    def close(self):
        if getattr(self, "_handle", None) is not None:
            self._lib.rvb_policy_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- forward
    def _forward(self, states, out=None):
        return _launch(self, None, states, out, None)[0]


def _packed(states, nets):
    """The packed form of `states`, (proprio, heightmap), checked against every network of `nets`; nothing is copied."""
    proprio, heightmap = packed_obs(states, max(n.num_proprioception for n in nets), max(n.num_exteroceptive for n in nets))
    _lib.require_cuda(proprio, heightmap)
    return proprio, heightmap


def packed_obs(states, p, e, what="states"):
    """`states` checked as the fused step's packed observation (proprio f32 [N, >=p], heightmap f16 [N, >=e]), e.g.
    `(task.obs_buf[:, :4], task.obs16_buf)`; returns the two tensors, nothing is copied (their device is the caller's to check).
    Shared by the networks and the teacher-data recorder (hooks.TeacherRecorder)."""
    form = ("packed %s must be (proprio float32 [N, >=%d], heightmap float16 [N, >=%d]) on one device, each with unit column "
            "stride" % (what, p, e))
    if len(states) != 2 or not all(isinstance(t, torch.Tensor) for t in states):
        raise RuntimeError(form)
    proprio, heightmap = states
    if (proprio.dim() != 2 or heightmap.dim() != 2 or proprio.dtype != torch.float32 or heightmap.dtype != torch.float16
            or proprio.shape[0] != heightmap.shape[0] or proprio.shape[1] < p or heightmap.shape[1] < e
            or proprio.stride(1) != 1 or heightmap.stride(1) != 1 or proprio.device != heightmap.device):
        raise RuntimeError(form)
    return proprio, heightmap


def _row_stride(t):
    return t.stride(0) if t.shape[0] > 1 else t.shape[1]     # a single row's stride is arbitrary in torch


def _launch(a, b, states, out_a, out_b):
    """Network a alone (b None) or the pair a, b on `states`: an f32 tensor [N, >=p+S+D] (rvb_policy_forward / _pair) or the packed
    2-tuple (proprio f32 [N, >=p], heightmap f16 [N, >=S+D]) (rvb_policy_forward_packed)."""
    nets = (a,) if b is None else (a, b)
    packed = isinstance(states, tuple)
    if packed:
        proprio, heightmap = _packed(states, nets)
        ref = proprio
    else:
        if isinstance(states, torch.Tensor):
            _lib.require_cuda(states)
        for net in nets:
            if not isinstance(states, torch.Tensor) or states.dim() != 2 or states.dtype != torch.float32 or states.shape[1] < net.num_observations:
                raise RuntimeError("states must be float32 [N, >=%d] or the packed 2-tuple (proprio float32 [N, >=%d], heightmap "
                                   "float16 [N, >=%d])" % (net.num_observations, net.num_proprioception, net.num_exteroceptive))
        if states.stride(1) != 1:
            states = states.contiguous()
        ref = states
    for net in nets:
        if net.device.index is not None and ref.device.index != net.device.index:
            raise RuntimeError("states live on %s, the network on %s" % (ref.device, net.device))
    N = ref.shape[0]
    if out_a is None:
        out_a = torch.empty((N, a._head_out), dtype=torch.float32, device=ref.device)
    if b is not None and out_b is None:
        out_b = torch.empty((N, b._head_out), dtype=torch.float32, device=ref.device)
    lib = a._lib
    with torch.cuda.device(ref.device):
        if packed:
            _lib.check(lib.rvb_policy_forward_packed(a._handle, None if b is None else b._handle, _lib.ptr(proprio), _row_stride(proprio),
                                                     _lib.ptr(heightmap), _row_stride(heightmap), N, _lib.ptr(out_a), out_a.stride(0),
                                                     _lib.ptr(out_b), 0 if b is None else out_b.stride(0), _lib.stream_of(ref)))
        elif b is None:
            _lib.check(lib.rvb_policy_forward(a._handle, _lib.ptr(states), states.stride(0), N, _lib.ptr(out_a), out_a.stride(0),
                                              _lib.stream_of(states)))
        else:
            _lib.check(lib.rvb_policy_forward_pair(a._handle, b._handle, _lib.ptr(states), states.stride(0), N, _lib.ptr(out_a),
                                                   out_a.stride(0), _lib.ptr(out_b), out_b.stride(0), _lib.stream_of(states)))
    return out_a, out_b


def compute_pair(policy, value, states, out_policy=None, out_value=None):
    """`policy.compute(states)[0]` and `value.compute(states)` in ONE launch (rvb_policy_forward_pair): the two calls a PPO
    step makes on the same states (skrl's agent.act + value.act on the reference's models_ppo, train.py:98-99).  `states` is the
    f32 observation or the step's packed form `(task.obs_buf[:, :4], task.obs16_buf)` (rvb_policy_forward_packed), which gives
    the same bits as its widened f32 rows without widening them."""
    return _launch(policy, value, states, out_policy, out_value)


class StochasticActorHeightmap(_HeightmapNet):
    """model.py:152-195: `compute()` returns (tanh(mean actions) f32[N, A], log_std_parameter f32[A])."""

    def __init__(self, observation_space, action_space, networkInfo, observartionInfo, device='cuda:0', clip_actions=False,
                 clip_log_std=True, min_log_std=-20.0, max_log_std=2.0, reduction="sum"):
        self.num_actions = _space_dim(action_space)
        super().__init__(observation_space, self.num_actions, networkInfo, observartionInfo, device, head_tanh=True)
        self.log_std_parameter = torch.zeros(self.num_actions, device=self.device)     # model.py:178

    def _extra_state(self):
        return {"log_std_parameter": self.log_std_parameter.detach().cpu().clone()}

    def _load_extra(self, sd):
        if "log_std_parameter" in sd:
            self.log_std_parameter = torch.as_tensor(sd["log_std_parameter"]).detach().to(self.device, torch.float32).clone()

    def compute(self, states, taken_actions=None, role=""):
        return self._forward(states), self.log_std_parameter


class DeterministicHeightmap(_HeightmapNet):
    """model.py:197-241: `compute()` returns the value f32[N, 1]."""

    def __init__(self, observation_space, action_space, networkInfo, observartionInfo, device='cuda:0', clip_actions=False):
        super().__init__(observation_space, 1, networkInfo, observartionInfo, device, head_tanh=False)

    def compute(self, states, taken_actions=None, role=""):
        return self._forward(states)
