"""The teacher-data recorder on the fused step's packed observation: rvb_teacher_record_packed bit for bit against rvb_teacher_record on
the widened rows and against the oracle (tests/teacher_packed_ref.py), the fused step's recorder fed from obs16_buf, the file of a
packed block and its device memory."""
import ctypes as C

import pytest
import torch

import teacher_packed_ref as TR

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import isaac_rover_b200
    return isaac_rover_b200


@pytest.fixture(scope="module")
def world20(R):
    return R.synth.make_world(length=20.0, nv=72, K=200, n_stones=12, seed=1)


def _ld(t):
    return t.stride(0) if t.shape[0] > 1 else t.shape[1]


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _inputs(n, p, e, layout, seed):
    """Device inputs of one recorder call.  layout "tight": contiguous rows.  "odd": the heightmap starts 2 bytes into a row of odd
    stride, proprio is the strided view obs[:, :p] of wider rows, actions have a row stride of 5 (see _outputs for the record
    rows)."""
    g = torch.Generator().manual_seed(seed)
    reset = torch.randn(n, generator=g)
    reset[::3] = 1.0
    if layout == "tight":
        actions = torch.randn(n, 2, generator=g).to(DEV)
        proprio = torch.randn(n, p, generator=g).to(DEV)
        hm = TR.heightmap_bits(n, e, seed).to(DEV).view(torch.float16)
    else:
        actions = torch.randn(n, 5, generator=g).to(DEV)[:, 1:3]
        proprio = torch.randn(n, p + 6, generator=g).to(DEV)[:, :p]
        hm = torch.zeros((n, e + 3), dtype=torch.int16, device=DEV)
        hm[:, 1:e + 1] = TR.heightmap_bits(n, e, seed).to(DEV)
        hm = hm.view(torch.float16)[:, 1:e + 1]
    return reset.to(DEV), actions, proprio, hm


def _outputs(n, p, e, layout, split):
    """(rec, rec16, rec_buf, rec16_buf): the record rows, views into sentinel-filled buffers whose other elements must stay.  Layout
    "odd": the rows start one element in, with strides 3 elements longer than the rows (1749 halves for the shipped heightmap)."""
    pad = 0 if layout == "tight" else 1
    width = 3 + p + (0 if split else e)
    rec_buf = torch.full((n, width + 2 * pad + (0 if layout == "tight" else 1)), -7.25, device=DEV)
    rec = rec_buf[:, pad:pad + width]
    rec16_buf = rec16 = None
    if split:
        rec16_buf = torch.full((n, e + 2 * pad + (0 if layout == "tight" else 1)), 0x5A5A, dtype=torch.int16, device=DEV)
        rec16 = rec16_buf[:, pad:pad + e]
    return rec, rec16, rec_buf, rec16_buf


def _record_packed(lib, reset, actions, proprio, hm, rec, rec16):
    p, e, n = proprio.shape[1], hm.shape[1], hm.shape[0]
    rc = lib.rvb_teacher_record_packed(_ptr(reset), _ptr(actions), _ld(actions), _ptr(proprio), _ld(proprio), p, _ptr(hm), _ld(hm), e,
                                       n, _ptr(rec), _ld(rec), _ptr(rec16), 0 if rec16 is None else _ld(rec16),
                                       C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, lib.rvb_last_error()


def _widened_reference(lib, reset, actions, proprio, hm):
    """rvb_teacher_record on the widened rows cat(proprio, heightmap.float()) (the widening done by torch on the device)."""
    obs = torch.cat([proprio, hm.float()], 1)
    n, c = obs.shape
    out = torch.empty((n, 3 + c), device=DEV)
    rc = lib.rvb_teacher_record(_ptr(reset), _ptr(actions), _ld(actions), _ptr(obs), _ld(obs), n, c, _ptr(out), _ld(out),
                                C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, lib.rvb_last_error()
    return out


def _check_call(R, n, p, e, layout, seed, oracle):
    lib = R._lib.load()
    reset, actions, proprio, hm = _inputs(n, p, e, layout, seed)
    ref = _widened_reference(lib, reset, actions, proprio, hm)
    rec, _, rec_buf, _ = _outputs(n, p, e, layout, split=False)
    before = rec_buf.clone()
    _record_packed(lib, reset, actions, proprio, hm, rec, None)
    head, rec16, head_buf, rec16_buf = _outputs(n, p, e, layout, split=True)
    before16, before_head = rec16_buf.clone(), head_buf.clone()
    _record_packed(lib, reset, actions, proprio, hm, head, rec16)
    torch.cuda.synchronize()
    # widened: the bits of rvb_teacher_record on cat(proprio, heightmap.float()); nothing outside the rows is written
    assert TR.same_bits(rec, ref)
    rec.fill_(-7.25)
    assert TR.same_bits(rec_buf, before)
    # split: the lead columns of the same rows, and every heightmap bit copied
    assert TR.same_bits(head, ref[:, :3 + p])
    assert torch.equal(rec16, hm.view(torch.int16))
    head.fill_(-7.25)
    rec16.fill_(0x5A5A)
    assert TR.same_bits(head_buf, before_head) and torch.equal(rec16_buf, before16)
    if oracle:                                      # the recorder's oracle on the host: every bit but NaN payloads
        rows, ohead, obits = TR.reference(reset.cpu(), actions.cpu(), proprio.cpu(), hm.cpu())
        assert TR.equal_but_nan_payloads(ref.cpu(), rows)
        assert TR.same_bits(ref[:, :3 + p].cpu(), ohead) and torch.equal(hm.view(torch.int16).cpu(), obits)
    del ref, rec, rec_buf, head, rec16, head_buf, rec16_buf, before, before16, hm
    torch.cuda.empty_cache()


@pytest.mark.parametrize("layout", ["tight", "odd"])
@pytest.mark.parametrize("n", [1, 31, 4096, 65535, 65536 + 7, 131072])
def test_kernel_bits_at_the_shipped_row(R, n, layout):
    _check_call(R, n, 4, 1746, layout, seed=n, oracle=n <= 4096)


@pytest.mark.parametrize("layout", ["tight", "odd"])
@pytest.mark.parametrize("p,e", [(0, 1), (0, 5), (4, 7), (8, 8), (8, 1745), (3, 2040), (4, 2041), (1, 4500)])
def test_kernel_bits_at_other_shapes(R, p, e, layout):
    _check_call(R, 37, p, e, layout, seed=100 * p + e, oracle=True)


def test_kernel_alignment_combinations(R):
    """Every start of the heightmap and of the fp16 record within a 16-byte line (and row strides of every residue), so the staged
    copy runs with the source and destination aligned alike and differently, and the f32 rows start at every residue too."""
    lib = R._lib.load()
    n, p, e = 9, 4, 1746
    bits = TR.heightmap_bits(n, e, 5).to(DEV)
    g = torch.Generator().manual_seed(6)
    reset, actions, proprio = (torch.randn(n, generator=g).to(DEV), torch.randn(n, 2, generator=g).to(DEV),
                               torch.randn(n, p, generator=g).to(DEV))
    for sh in range(8):
        for extra in (0, 1, 2, 5):
            src = torch.zeros((n, e + 8 + extra), dtype=torch.int16, device=DEV)
            src[:, sh:sh + e] = bits
            hm = src.view(torch.float16)[:, sh:sh + e]
            ref = _widened_reference(lib, reset, actions, proprio, hm)
            for dsh in (0, 1, 3, 6):
                dst = torch.zeros((n, e + 8 + extra), dtype=torch.int16, device=DEV)
                head = torch.empty((n, 3 + p + dsh), device=DEV)[:, dsh:]
                _record_packed(lib, reset, actions, proprio, hm, head, dst[:, dsh:dsh + e])
                wide = torch.zeros((n, 3 + p + e + 4 + extra), device=DEV)
                _record_packed(lib, reset, actions, proprio, hm, wide[:, dsh % 4:dsh % 4 + 3 + p + e], None)
                assert torch.equal(dst[:, dsh:dsh + e], bits), (sh, extra, dsh)
                assert TR.same_bits(head, ref[:, :3 + p]) and TR.same_bits(wide[:, dsh % 4:dsh % 4 + 3 + p + e], ref), (sh, extra, dsh)


def test_widening_equals_torch_float_on_the_device(R):
    """Every one of the 65,536 fp16 bit patterns widened by the kernel equals torch's .float() on the device, NaN payloads included;
    the split form copies every pattern."""
    lib = R._lib.load()
    allbits = torch.arange(-32768, 32768, dtype=torch.int32).to(torch.int16).reshape(32, 2048).to(DEV)
    hm = allbits.view(torch.float16)
    n = hm.shape[0]
    zeros = torch.zeros(n, device=DEV)
    acts = torch.zeros((n, 2), device=DEV)
    rec = torch.empty((n, 3 + hm.shape[1]), device=DEV)
    _record_packed(lib, zeros, acts, torch.empty((n, 0), device=DEV), hm, rec, None)
    head, rec16 = torch.empty((n, 3), device=DEV), torch.empty_like(allbits)
    _record_packed(lib, zeros, acts, torch.empty((n, 0), device=DEV), hm, head, rec16)
    torch.cuda.synchronize()
    assert TR.same_bits(rec[:, 3:], hm.float())
    assert torch.equal(rec16, allbits)
    kept = torch.equal(rec[:, 3:].cpu().view(torch.int32), hm.cpu().float().view(torch.int32))
    print("device widening keeps NaN payloads like the host's: %s" % kept)


# ---------------------------------------------------------------- the fused step's recorder in packed mode
def _physics(views, k):
    """Stand-in for the simulator's step between the halves: the same pose and joint change for every view."""
    g = torch.Generator().manual_seed(700 + k)
    n = views[0].pos.shape[0]
    dpos = ((torch.rand(n, 3, generator=g) - 0.5) * 0.2).cuda()
    dq = ((torch.rand(n, 4, generator=g) - 0.5) * 0.3).cuda()
    dj = ((torch.rand(n, 13, generator=g) - 0.5) * 0.1).cuda()
    for v in views:
        v.pos = (v.pos + dpos).contiguous()
        q = v.quat + dq
        v.quat = (q / q.norm(dim=1, keepdim=True)).contiguous()
        v.joints = (v.joints + dj).contiguous()


def _recording_tasks(R, world, n, steps, tmp_path):
    """Three tasks from the same world and poses: f32 observation + f32 recorder, packed observation + f32 recorder, packed
    observation + packed recorder."""
    st = R.synth.make_env_state(world, n, seed=61)
    tasks = []
    for name, obs16, packed in (("f32", False, False), ("obs16", True, False), ("packed", True, True)):
        t = R.synth.make_task(world, st, device=DEV, level=2)
        t.reset_buf.zero_()
        t.reset_buf[::7] = 1
        if obs16:
            t.obs16_buf = torch.zeros((n, t.num_observations - 4), dtype=torch.float16, device=DEV)
        hm = t.Camera.heightmap
        d = tmp_path / name
        d.mkdir()
        t.save_teacher_data = True
        t.teacher_recorder = R.TeacherRecorder(n, t.num_observations, hm.get_num_sparse_vector(), hm.get_num_dense_vector(),
                                               steps=steps, directory=str(d), packed=packed)
        tasks.append(t)
    return tasks


def _blocks_equal(tasks, k):
    """The first k timesteps of the three recorders: torch.equal, the packed block after widening."""
    f32, obs16, packed = (t.teacher_recorder for t in tasks)
    a = f32.teacher_dataset[:k]
    assert torch.equal(obs16.teacher_dataset[:k], a)
    widened = torch.stack([packed.widened_step(t) for t in range(k)])
    assert torch.equal(widened, a)
    assert torch.equal(packed.teacher_heightmap[:k].float(), a[:, :, 7:]) and torch.equal(packed.teacher_head[:k], a[:, :, :7])
    # the rows hold real observations: resets flagged, heightmap columns of the earlier steps' observations
    assert bool((a[1:, :, 0] == 1).any()) and bool((a[1:, :, 7:] != 0).any())
    return a


def _files_equal(tasks):
    saved = [torch.load(t.teacher_recorder.last_file) for t in tasks]
    for s in saved[1:]:
        assert s["info"] == saved[0]["info"]
        assert s["data"].dtype == torch.float32 and s["data"].shape == saved[0]["data"].shape
        assert torch.equal(s["data"], saved[0]["data"])
    assert saved[0]["info"] == {"reset": 1, "actions": 2, "proprioceptive": 4, "sparse": 634, "dense": 1112}
    return saved[0]["data"]


def test_hot_step_records_the_packed_observation(R, world20, tmp_path):
    """hot_step(device_reset=True) with obs16_buf: the recorder rows are those of the f32 run (at the parent commit the obs16_buf
    task recorded the never-written obs_buf[:, 4:]), for an f32 and a packed recorder, and the files they write are equal."""
    n, steps = 300, 6
    tasks = _recording_tasks(R, world20, n, steps, tmp_path)
    g = torch.Generator().manual_seed(9)
    for k in range(steps):
        act = (torch.rand(n, 2, generator=g) * 2 - 1).cuda()
        for t in tasks:
            t.hot_step(act, device_reset=True)
        torch.cuda.synchronize()
        if k == steps - 2:
            _blocks_equal(tasks, steps - 1)
        assert torch.equal(tasks[1].obs16_buf.float(), tasks[0].obs_buf[:, 4:])
    data = _files_equal(tasks)
    assert data.shape == (steps, n, 1753)


def test_fused_halves_record_the_packed_observation(R, world20, tmp_path):
    """pre_physics_step_fused + post_physics_step_fused with a pose change between the halves: the same rows and files."""
    n, steps = 300, 5
    tasks = _recording_tasks(R, world20, n, steps, tmp_path)
    g = torch.Generator().manual_seed(10)
    for k in range(steps):
        act = (torch.rand(n, 2, generator=g) * 2 - 1).cuda()
        for t in tasks:
            t.pre_physics_step_fused(act)
        _physics([t._rover for t in tasks], k)
        for t in tasks:
            t.post_physics_step_fused()
        torch.cuda.synchronize()
        if k == steps - 2:
            _blocks_equal(tasks, steps - 1)
    _files_equal(tasks)


def test_packed_recorder_refuses_the_f32_observation_of_a_task(R, world20):
    st = R.synth.make_env_state(world20, 16, seed=62)
    t = R.synth.make_task(world20, st, device=DEV, level=1)
    t.save_teacher_data = True
    t.teacher_recorder = R.TeacherRecorder(16, t.num_observations, 634, 1112, steps=2, save=False, packed=True)
    with pytest.raises(RuntimeError, match="records the packed observation"):
        t.hot_step(torch.zeros(16, 2, device=DEV))


# ---------------------------------------------------------------- device memory
def test_packed_block_is_half_the_device_memory(R):
    n, steps = 4096, 150
    sizes = {}
    for packed in (False, True):
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        rec = R.TeacherRecorder(n, 1750, 634, 1112, steps=steps, save=False, packed=packed)
        sizes[packed] = torch.cuda.memory_allocated() - before
        del rec
    print("device block at %d envs x %d steps: f32 %.3f GB, packed %.3f GB" % (n, steps, sizes[False] / 1e9, sizes[True] / 1e9))
    assert abs(sizes[False] - steps * n * 7012) <= 4096
    assert abs(sizes[True] - steps * n * 3520) <= 4096
    assert abs(sizes[False] / 1e9 - 4.31) < 0.01 and abs(sizes[True] / 1e9 - 2.16) < 0.01
