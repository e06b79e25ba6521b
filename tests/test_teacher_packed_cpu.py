"""The teacher-data recorder on the packed observation (rvb_teacher_record_packed, TeacherRecorder(packed=...)): the checks that run
on the host before anything touches a device, and the reference the GPU tests hold the kernel to."""
import ctypes

import pytest
import torch

import teacher_packed_ref as TR

E, P = 1746, 4


def _call(lib, reset=True, actions=True, actions_ld=2, proprio=True, proprio_ld=4, p=P, heightmap=True, heightmap_ld=E, e=E, n=4,
          rec=True, rec_ld=3 + P + E, rec16=False, rec16_ld=E):
    """One call with host buffers standing in for the device arrays: every case below is refused before the kernel could read them."""
    f = lambda k: (ctypes.c_float * k)()
    h = lambda k: (ctypes.c_uint16 * k)()
    args = (f(16) if reset else None, f(16) if actions else None, actions_ld, f(16) if proprio else None, proprio_ld, p,
            h(16) if heightmap is True else heightmap or None, heightmap_ld, e, n, f(16) if rec else None, rec_ld,
            h(16) if rec16 else None, rec16_ld, None)
    return lib.rvb_teacher_record_packed(*args)


@pytest.fixture(scope="module")
def lib():
    import isaac_rover_b200
    from isaac_rover_b200 import _lib
    return _lib.load()


def _refused(lib, rc, what):
    assert rc == -1, rc
    assert ("rvb_teacher_record_packed: " + what).encode() in lib.rvb_last_error(), lib.rvb_last_error()


@pytest.mark.parametrize("missing", ["reset", "actions", "proprio", "heightmap", "rec"])
def test_entry_point_refuses_null_pointers(lib, missing):
    _refused(lib, _call(lib, **{missing: False}), "null pointer")


def test_null_proprio_is_allowed_without_proprioceptive_columns(lib):
    # p == 0 passes the pointer check; the call is then refused for its short record row, not for the null proprio
    _refused(lib, _call(lib, proprio=False, p=0, proprio_ld=0, rec_ld=2), "short row")


def test_zero_rows_is_a_no_op(lib):
    assert lib.rvb_teacher_record_packed(None, None, 2, None, 4, 4, None, E, E, 0, None, 3 + P + E, None, E, None) == 0


@pytest.mark.parametrize("p", [-1, 9, 100])
def test_entry_point_refuses_p_outside_0_to_8(lib, p):
    _refused(lib, _call(lib, p=p, proprio_ld=max(p, 4), rec_ld=3 + max(p, 0) + E), "p must be in 0..8")


@pytest.mark.parametrize("kw", [dict(e=0, heightmap_ld=0, rec_ld=3 + P), dict(e=-3), dict(n=-1), dict(e=1 << 30, heightmap_ld=1 << 30,
                                                                                                        rec_ld=(1 << 30) + 7)])
def test_entry_point_refuses_bad_shapes(lib, kw):
    _refused(lib, _call(lib, **kw), "bad shape")


SHORT = {
    "actions_ld": dict(actions_ld=1),
    "proprio_ld": dict(proprio_ld=3),
    "heightmap_ld": dict(heightmap_ld=E - 1),
    "rec_ld_widened": dict(rec_ld=3 + P + E - 1),
    "rec_ld_split": dict(rec16=True, rec_ld=3 + P - 1),
    "rec16_ld": dict(rec16=True, rec_ld=3 + P, rec16_ld=E - 1),
    "rec_ld_p8": dict(p=8, proprio_ld=8, rec_ld=3 + 4 + E),
}


@pytest.mark.parametrize("what", sorted(SHORT))
def test_entry_point_refuses_short_rows(lib, what):
    _refused(lib, _call(lib, **SHORT[what]), "short row")


def test_entry_point_refuses_misaligned_pointers(lib):
    buf = (ctypes.c_uint16 * 32)()
    odd = ctypes.c_void_p(ctypes.addressof(buf) + 1)
    _refused(lib, _call(lib, heightmap=odd), "misaligned pointer")


# ---------------------------------------------------------------- TeacherRecorder: refusals on the host
def _unbuilt(packed, n=5):
    """A recorder as far as the host-side checks see it (no device block: nothing here may reach the library)."""
    import isaac_rover_b200 as R
    rec = object.__new__(R.TeacherRecorder)
    rec.num_envs, rec.num_observations, rec.num_proprioceptive, rec.packed = n, 1750, 4, packed
    return rec


def test_packed_recorder_refuses_f32_rows():
    rec = _unbuilt(True)
    for obs in (torch.zeros(5, 1750), torch.zeros(5, 1750).half()):
        with pytest.raises(RuntimeError, match=r"records the packed observation .* only, not float32 rows: .*fp16"):
            rec.record(torch.zeros(5), torch.zeros(5, 2), obs)


BAD = {
    "heightmap_f32": lambda N: (torch.zeros(N, 4), torch.zeros(N, 1746)),
    "proprio_f16": lambda N: (torch.zeros(N, 4, dtype=torch.float16), torch.zeros(N, 1746, dtype=torch.float16)),
    "proprio_narrow": lambda N: (torch.zeros(N, 3), torch.zeros(N, 1746, dtype=torch.float16)),
    "heightmap_narrow": lambda N: (torch.zeros(N, 4), torch.zeros(N, 1745, dtype=torch.float16)),
    "heightmap_column_stride": lambda N: (torch.zeros(N, 4), torch.zeros(N, 3492, dtype=torch.float16)[:, ::2]),
    "row_count_mismatch": lambda N: (torch.zeros(N, 4), torch.zeros(N + 1, 1746, dtype=torch.float16)),
    "three_items": lambda N: (torch.zeros(N, 4), torch.zeros(N, 1746, dtype=torch.float16), torch.zeros(N, 4)),
    "not_tensors": lambda N: ([0.0] * 4, [0.0] * 1746),
}


@pytest.mark.parametrize("packed", [False, True])
@pytest.mark.parametrize("what", sorted(BAD))
def test_recorder_refuses_a_malformed_packed_tuple(what, packed):
    rec = _unbuilt(packed)
    with pytest.raises(RuntimeError, match=r"packed obs must be \(proprio float32 \[N, >=4\], heightmap float16 \[N, >=1746\]\)"):
        rec.record(torch.zeros(5), torch.zeros(5, 2), BAD[what](5))


@pytest.mark.parametrize("packed", [False, True])
def test_recorder_refuses_a_pair_of_other_rows(packed):
    rec = _unbuilt(packed, n=6)
    with pytest.raises(RuntimeError, match="packed obs must have 6 rows"):
        rec.record(torch.zeros(6), torch.zeros(6, 2), (torch.zeros(5, 4), torch.zeros(5, 1746, dtype=torch.float16)))


def test_f32_recorder_names_both_forms_and_has_no_cpu_path():
    rec = _unbuilt(False)
    with pytest.raises(RuntimeError, match=r"obs must be float32 \[5, >=1750\] or the packed pair"):
        rec.record(torch.zeros(5), torch.zeros(5, 2), [torch.zeros(5, 4), torch.zeros(5, 1746, dtype=torch.float16)])
    with pytest.raises(RuntimeError, match=r"obs must be float32 \[5, >=1750\]"):
        rec.record(torch.zeros(5), torch.zeros(5, 2), torch.zeros(5, 1749))
    for packed in (False, True):                      # well-formed, but on the host: there is no CPU path
        with pytest.raises(RuntimeError, match="expected a CUDA tensor"):
            _unbuilt(packed).record(torch.zeros(5), torch.zeros(5, 2), (torch.zeros(5, 4), torch.zeros(5, 1746, dtype=torch.float16)))


def test_recorder_needs_a_cuda_device():
    import isaac_rover_b200 as R
    with pytest.raises(RuntimeError, match="needs a CUDA device"):
        R.TeacherRecorder(4, 1750, 634, 1112, device="cpu", packed=True)


# ---------------------------------------------------------------- the reference of both modes
def test_reference_rows_are_the_oracle_rows_of_the_widened_observation():
    n, p, e = 23, 4, 1746
    g = torch.Generator().manual_seed(7)
    reset = (torch.rand(n, generator=g) < 0.5).float()
    actions = torch.rand(n, 2, generator=g) * 2 - 1
    proprio = torch.randn(n, p, generator=g)
    bits = TR.heightmap_bits(n, e, seed=8)
    hm = bits.view(torch.float16)
    rows, head, hbits = TR.reference(reset, actions, proprio, hm)
    # the reference's statement (rover.py:299): cat(reset_info, actions, obs_buf), obs_buf holding the heightmap as f32 values
    literal = torch.cat([reset[:, None], actions, proprio, hm.float()], 1)
    assert TR.same_bits(rows, literal)
    assert TR.same_bits(head, rows[:, :3 + p]) and torch.equal(hbits, bits)
    # fp16 -> f32 is exact: the split form holds every bit of the widened row, special values included
    assert TR.same_bits(torch.cat([head, hbits.view(torch.float16).float()], 1), rows)
    assert torch.equal(rows[:, 3 + p:].half().view(torch.int16)[~torch.isnan(rows[:, 3 + p:])], bits[~torch.isnan(hm)])
    v = hm.float()
    assert bool(torch.isnan(v).any() and torch.isinf(v).any() and ((v != 0) & (v.abs() < 2.0 ** -14)).any())
    assert bool((bits == 0).any() and (bits == -32768).any())                # +0 and -0
