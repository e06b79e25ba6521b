"""The C-ABI library builds, loads, and exports every symbol include/rover_b200.h declares (no compute)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "rover_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rvb_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported_abi5():
    import isaac_rover_b200
    from isaac_rover_b200 import _lib
    lib = _lib.load()
    names = declared_symbols()
    assert len(names) >= 20
    raw = ctypes.CDLL(_lib.lib_path())
    for n in names:
        assert hasattr(raw, n), "missing export " + n
    assert set(names) == set(_lib.EXPORTS), set(names) ^ set(_lib.EXPORTS)
    for n in ("rvb_terrain_create", "rvb_heightmap_raycast", "rvb_rock_collision"):        # their "2" forms were merged into them
        assert not hasattr(raw, n + "2"), "removed entry point still exported: " + n + "2"
    assert not hasattr(raw, "rvb_env_step"), "removed entry point still exported: rvb_env_step"    # the pair pre + post replaced it
    assert lib.rvb_abi_version() == 5


def test_argument_validation_without_gpu():
    """Host-side validation runs before any CUDA call, so it is testable on a CPU-only box."""
    import isaac_rover_b200
    from isaac_rover_b200 import _lib
    lib = _lib.load()
    rc = lib.rvb_quat_to_euler(None, 4, None, None)
    assert rc == -1 and b"null pointer" in lib.rvb_last_error()
    rc = lib.rvb_ackermann(None, 1, None, 1, 4, None, None, None, None, 0, None)
    assert rc == -1
    h = ctypes.c_void_p()
    rc = lib.rvb_terrain_create(ctypes.byref(h), None, 10, 10, 8, 1, 1, 1, None, 4, None, 4, 0.1, 0.0, 0.0, 0, 0, None)
    assert rc == -1 and h.value is None
    rc = lib.rvb_terrain_create(ctypes.byref(h), None, 10, 10, 8, 1, 1, 1, None, 4, None, 4, 0.1, 0.0, 0.0, 0, 2, None)
    assert rc == -1 and h.value is None and b"rvb_terrain_create: unknown flag" in lib.rvb_last_error()
    assert lib.rvb_heightmap_raycast(None, None, None, None, None, 4, 1, None, None, None, None, None,
                                     None, 0, None, 0, 0, None, None, 0, None) == -1
    assert lib.rvb_cast_rays(None, None, None, 4, None, None, None, None, None) == -1
    assert lib.rvb_rock_collision(None, None, None, None, None, None, 4, None, None, None, None, None, None) == -1
    assert lib.rvb_check_collision(None, None, 4, None, None) == -1
    # policy dispatch: 2 = default, 1 = FFMA2 kernel for every shape; the removed variants 0 and 3 are refused
    assert lib.rvb_policy_variant(-1) == 2
    for v in (0, 3):
        assert lib.rvb_policy_variant(v) == -1 and b"removed" in lib.rvb_last_error()
        assert lib.rvb_policy_variant(-1) == 2
    assert lib.rvb_policy_variant(1) == 2
    assert lib.rvb_policy_variant(2) == 1
    assert lib.rvb_policy_variant(-1) == 2
    assert lib.rvb_stats_scratch_len(1000) == 4 * 16
    # policy epilogue / hooks (SURVEY 8f-3, 8f-4)
    h = ctypes.c_void_p()
    rc = lib.rvb_policy_create(ctypes.byref(h), 4, 634, 1112, None, None, None, None, 0, 1, 0, None)
    assert rc == -1 and h.value is None and b"null pointer" in lib.rvb_last_error()
    lin = (_lib.Linear * 3)()
    rc = lib.rvb_policy_create(ctypes.byref(h), 9, 634, 1112, lin, lin, lin, lin, 0, 1, 0, None)      # more than 8 proprioceptive columns
    assert rc == -1 and h.value is None
    rc = lib.rvb_policy_create(ctypes.byref(h), 4, 634, 1112, lin, lin, lin, lin, 17, 1, 0, None)     # unknown activation
    assert rc == -1 and b"activation" in lib.rvb_last_error()
    assert lib.rvb_policy_forward(None, None, 1750, 4, None, 2, None) == -1
    assert lib.rvb_policy_forward_pair(None, None, None, 1750, 4, None, 2, None, 1, None) == -1
    assert lib.rvb_policy_destroy(None) == 0 and lib.rvb_policy_bytes(None) == 0
    assert lib.rvb_obs_hooks(None, 1750, 4, 1750, 4, 0.0, 0.0, 0.0, None, 1, 1, 0, None) == -1
    assert lib.rvb_obs_hooks(None, 1750, 0, 1750, 4, 0.0, 0.0, 0.0, None, 1, 1, 0, None) == 0        # nothing to do
    assert lib.rvb_teacher_record(None, None, 2, None, 1750, 4, 1750, None, 1753, None) == -1


def test_no_cpu_fallback():
    import torch
    import isaac_rover_b200 as R
    with pytest.raises(RuntimeError):
        R.tensor_quat_to_eul(torch.zeros(2, 4))
    with pytest.raises(RuntimeError):
        R.ray_distance(torch.zeros(4, 3), torch.zeros(4, 3), torch.zeros(4, 3, 3))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "isaac_rover_2.0_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "rover_oracle" not in text and "ref_import" not in text and "/root/reference" not in text, f
                assert "libray_oracle" not in text, f
                if f.endswith(".py"):                      # no import of anything under oracle/ (comments may cite it)
                    assert not re.search(r"^\s*(import|from)\s+\S*oracle", text, flags=re.M), f


def test_library_staleness_is_by_content_not_mtime(monkeypatch):
    """The built library travels to the GPU box in a copy of the tree (mtimes are not preserved) and eight ranks import it at
    once: staleness must be decided from a hash of the sources, never from timestamps."""
    import isaac_rover_b200
    from isaac_rover_b200 import _build
    assert os.path.exists(_build.LIB) and os.path.exists(_build.HASH_FILE)
    assert _build.needs_build() is False
    os.utime(_build.LIB, (1, 1))                                   # an ancient library with matching sources is still current
    assert _build.needs_build() is False
    monkeypatch.setattr(_build, "NVCC_FLAGS", _build.NVCC_FLAGS + ["-DSOMETHING"])
    assert _build.needs_build() is True                            # other flags (or sources) = another hash
