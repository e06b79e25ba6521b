"""The packed-observation policy call (rvb_policy_forward_packed, model.compute / compute_pair on (proprio, heightmap)): the
checks that run on the host before anything touches a device."""
import ctypes

import pytest
import torch


def test_entry_point_refuses_null_pointers_and_handles():
    import isaac_rover_b200
    from isaac_rover_b200 import _lib
    lib = _lib.load()
    assert lib.rvb_policy_forward_packed(None, None, None, 4, None, 1746, 4, None, 2, None, 1, None) == -1
    assert b"rvb_policy_forward_packed: null pointer" in lib.rvb_last_error()
    # host buffers stand in for the device arrays: the call is refused before it reads them
    prop, hm, out_a, out_b = (ctypes.c_float * 16)(), (ctypes.c_uint16 * 16)(), (ctypes.c_float * 16)(), (ctypes.c_float * 16)()
    assert lib.rvb_policy_forward_packed(None, None, prop, 4, hm, 1746, 4, out_a, 2, None, 1, None) == -1
    assert b"rvb_policy_forward_packed: null handle" in lib.rvb_last_error()
    # a pair without out_b: refused as a null pointer whatever the handles are
    fake = (ctypes.c_char * 64)()
    assert lib.rvb_policy_forward_packed(fake, fake, prop, 4, hm, 1746, 4, out_a, 2, None, 1, None) == -1
    assert b"null pointer" in lib.rvb_last_error()
    assert lib.rvb_policy_forward_packed(None, None, None, 4, None, 1746, 0, None, 2, None, 1, None) == -1   # no handle, no rows
    assert b"null handle" in lib.rvb_last_error()


def _unbuilt(cls, n_head):
    """A network object as far as the host-side checks see it (no device handle: nothing here may reach the library)."""
    import isaac_rover_b200 as R
    net = object.__new__(cls)
    net.num_proprioception, net.num_sparse, net.num_dense = 4, 634, 1112
    net.num_exteroceptive, net.num_observations = 1746, 1750
    net.device, net._head_out, net._handle, net._lib = torch.device("cuda:0"), n_head, None, None
    net.log_std_parameter = torch.zeros(n_head)
    return net


BAD = {
    "heightmap_f32": lambda N: (torch.zeros(N, 4), torch.zeros(N, 1746)),
    "proprio_f16": lambda N: (torch.zeros(N, 4, dtype=torch.float16), torch.zeros(N, 1746, dtype=torch.float16)),
    "proprio_narrow": lambda N: (torch.zeros(N, 3), torch.zeros(N, 1746, dtype=torch.float16)),
    "heightmap_narrow": lambda N: (torch.zeros(N, 4), torch.zeros(N, 1745, dtype=torch.float16)),
    "proprio_column_stride": lambda N: (torch.zeros(N, 8)[:, ::2], torch.zeros(N, 1746, dtype=torch.float16)),
    "heightmap_column_stride": lambda N: (torch.zeros(N, 4), torch.zeros(N, 3492, dtype=torch.float16)[:, ::2]),
    "heightmap_transposed": lambda N: (torch.zeros(N, 4), torch.zeros(1746, N, dtype=torch.float16).t()),
    "row_count": lambda N: (torch.zeros(N, 4), torch.zeros(N + 1, 1746, dtype=torch.float16)),
    "heightmap_1d": lambda N: (torch.zeros(N, 4), torch.zeros(N * 1746, dtype=torch.float16)),
    "three_items": lambda N: (torch.zeros(N, 4), torch.zeros(N, 1746, dtype=torch.float16), torch.zeros(N, 4)),
    "not_tensors": lambda N: ([0.0] * 4, [0.0] * 1746),
}


@pytest.mark.parametrize("what", sorted(BAD))
def test_compute_rejects_a_malformed_packed_tuple(what):
    import isaac_rover_b200 as R
    actor = _unbuilt(R.model.StochasticActorHeightmap, 2)
    critic = _unbuilt(R.model.DeterministicHeightmap, 1)
    states = BAD[what](5)
    expected = r"packed states must be \(proprio float32 \[N, >=4\], heightmap float16 \[N, >=1746\]\)"
    for call in (lambda: actor.compute(states), lambda: critic.compute(states), lambda: R.model.compute_pair(actor, critic, states)):
        with pytest.raises(RuntimeError, match=expected):
            call()


def test_compute_names_both_forms_for_other_states():
    import isaac_rover_b200 as R
    actor = _unbuilt(R.model.StochasticActorHeightmap, 2)
    with pytest.raises(RuntimeError, match=r"states must be float32 \[N, >=1750\] or the packed 2-tuple"):
        actor.compute([torch.zeros(5, 4), torch.zeros(5, 1746, dtype=torch.float16)])
    with pytest.raises(RuntimeError, match="expected a CUDA tensor"):          # a well-formed pair on the host: no CPU path
        actor.compute((torch.zeros(5, 4), torch.zeros(5, 1746, dtype=torch.float16)))
