"""rvb_env_pre / rvb_env_post (the fused step split at the simulator's boundary) validate their arguments on the host before any
CUDA call, so a bad call is refused with RVB_ERR_INVALID and a message on a machine without a GPU too.  The pointers below are
never dereferenced: every call is refused before anything is launched."""
import ctypes

import pytest

FAKE = 0x10000          # 16-byte aligned, never read


@pytest.fixture(scope="module")
def lib():
    import isaac_rover_b200
    from isaac_rover_b200 import _lib
    return _lib.load()


def _pre(lib, quat=FAKE, actions=FAKE, N=4, H=3, lin=FAKE, ang=FAKE, rot=FAKE):
    return lib.rvb_env_pre(quat, actions, N, H, lin, ang, rot, None, None, 0, None)


def _io(**kw):
    from isaac_rover_b200 import _lib
    io = _lib.StepIO()
    for name, _ in _lib.StepIO._fields_:
        setattr(io, name, FAKE)
    io.obs_ld, io.obs_h16_ld = 1750, 0
    io.obs_h16 = None                                               # the packed observation is optional
    for name, v in kw.items():
        setattr(io, name, v)
    return io


def _post(lib, io, level=1, rocks=None, rot=FAKE, H=3, N=4):
    from isaac_rover_b200 import _lib
    prm = _lib.RewardParams(1.0, 0.05, -0.01, 0.3, 0.5, 3000, level, N, 0, 0)
    return lib.rvb_env_post(FAKE, rocks, ctypes.byref(prm), ctypes.byref(io), rot, FAKE, 1750, FAKE, FAKE, N, H, None)


def _refused(lib, rc, what):
    assert rc == -1, rc
    msg = lib.rvb_last_error()
    assert what in msg, msg


def test_env_pre_validation_abi5_without_gpu(lib):
    assert _pre(lib, N=0) == 0                                    # nothing to do
    _refused(lib, _pre(lib, N=-1), b"N < 0")
    for k in ("quat", "actions", "lin", "ang", "rot"):
        _refused(lib, _pre(lib, **{k: None}), b"rvb_env_pre: null pointer")
    _refused(lib, _pre(lib, quat=FAKE + 4), b"16-byte aligned")
    for H in (1, 65):
        _refused(lib, _pre(lib, H=H), b"history length")


def test_env_post_validation_without_gpu(lib):
    io = _io()
    assert lib.rvb_env_post(None, None, None, None, None, None, 1750, None, None, 0, 3, None) == 0     # nothing to do
    _refused(lib, _post(lib, io, N=-1), b"N < 0")
    _refused(lib, _post(lib, io, rot=None), b"rvb_env_post: null pointer")
    _refused(lib, lib.rvb_env_post(FAKE, None, None, ctypes.byref(io), FAKE, FAKE, 1750, FAKE, FAKE, 4, 3, None), b"null pointer")
    for k in ("pos", "quat", "joints", "target", "lin_hist", "ang_hist", "euler", "heading", "obs", "dist", "rew", "reset", "progress"):
        _refused(lib, _post(lib, _io(**{k: None})), b"null pointer in rvb_step_io")
    _refused(lib, _post(lib, _io(quat=FAKE + 8)), b"16-byte aligned")
    for H in (1, 65):
        _refused(lib, _post(lib, io, H=H), b"bad history length")
    _refused(lib, _post(lib, _io(obs_ld=3)), b"bad history length or obs_ld")
    _refused(lib, _post(lib, _io(obs_h16=FAKE)), b"obs_h16 needs obs_h16_ld")
    _refused(lib, _post(lib, io, level=2), b"rock layer")                        # curriculum level 2 without the rock layer
    _refused(lib, _post(lib, _io(wheel_dist=None), level=2, rocks=FAKE), b"rock layer")
