"""Reference rows of the teacher-data recorder on the packed observation (rvb_teacher_record_packed), built on the recorder's oracle
(oracle/hooks_oracle.teacher_row): the widened row is teacher_row(reset_info, actions, cat(proprio, heightmap.float())); the split
form is that row's first 3 + p columns plus the heightmap's fp16 bits, unchanged.  Shared by the CPU and the GPU tests."""
import torch

import hooks_oracle as HO

# fp16 bit patterns every kernel test mixes in: +0, -0, the smallest and largest subnormals of both signs, the smallest normal,
# the largest finite, +inf, -inf, the quiet NaN, signalling NaNs, NaNs with payloads of both signs, the all-ones NaN
SPECIAL_BITS = (0x0000, 0x8000, 0x0001, 0x8001, 0x03FF, 0x83FF, 0x0400, 0x7BFF, 0x7C00, 0xFC00, 0x7E00, 0x7C01, 0x7D55, 0xFE01,
                0xFFFF, 0x7FFF)


def heightmap_bits(n, e, seed):
    """int16 [n, e] of fp16 bit patterns: every pattern equally likely (NaNs and subnormals included), SPECIAL_BITS spread over
    every row."""
    g = torch.Generator().manual_seed(seed)
    bits = torch.randint(-32768, 32768, (n, e), generator=g, dtype=torch.int32)
    sp = torch.tensor(SPECIAL_BITS, dtype=torch.int32)
    sp = torch.where(sp >= 32768, sp - 65536, sp)
    cols = torch.arange(min(e, len(SPECIAL_BITS)))
    bits[:, (cols * 7) % e] = sp[cols]
    return bits.to(torch.int16)


def reference(reset_info, actions, proprio, heightmap):
    """CPU tensors (heightmap f16) -> (rows f32 [N, 3 + p + E], head f32 [N, 3 + p], heightmap bits int16 [N, E])."""
    obs = torch.cat([proprio.float(), heightmap.float()], 1)
    rows = torch.from_numpy(HO.teacher_row(reset_info.numpy(), actions.numpy(), obs.numpy()))
    p = proprio.shape[1]
    return rows, rows[:, :3 + p].clone(), heightmap.view(torch.int16).clone()


def same_bits(a, b):
    """Bit equality of two f32 tensors (NaN payloads included)."""
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def equal_but_nan_payloads(a, b):
    """Bit equality where b is not NaN, NaN where b is NaN: a widening done on the device may or may not keep a NaN's payload."""
    nan = torch.isnan(b)
    return bool(torch.isnan(a)[nan].all()) and torch.equal(a.view(torch.int32)[~nan], b.view(torch.int32)[~nan])
