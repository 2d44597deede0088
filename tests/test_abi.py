"""The C-ABI library loads and exports every symbol include/d2d_b200.h declares (no compute, no GPU)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "d2d_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(d2d_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from d2d_ppo_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "build the library first: python -c 'import __graft_entry__ as g; g.build()'"
    handle = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in d2d_b200.h but not exported"


def test_binding_covers_header():
    from d2d_ppo_b200 import _lib
    assert set(_lib.exported_symbols()) == set(_declared())


def test_version_and_error_string():
    from d2d_ppo_b200 import _lib
    lib = _lib.lib()
    assert lib.d2d_abi_version() == 1
    assert isinstance(lib.d2d_last_error(), bytes)
    # argument validation happens before any CUDA call, so it is checkable without a GPU
    assert lib.d2d_env_create(None, None) == _lib.ERR_INVALID
    assert b"null" in lib.d2d_last_error()


def test_kernel_switch_ids():
    """The header's D2D_SWITCH_* ids are the binding's; any other id is rejected (no CUDA is touched)."""
    from d2d_ppo_b200 import _lib
    src = open(os.path.join(ROOT, "include", "d2d_b200.h")).read()
    declared = {k: int(v) for k, v in re.findall(r"#define D2D_(SWITCH_\w+)\s+(\d+)", src)}
    assert declared == {k: getattr(_lib, k) for k in ("SWITCH_ALL_TC", "SWITCH_ENV_MULTISTEP", "SWITCH_HOST_PACK")}
    lib = _lib.lib()
    for which in declared.values():
        on = lib.d2d_get_kernel_switch(which)
        assert on in (0, 1)
        assert lib.d2d_set_kernel_switch(which, on) == _lib.OK and lib.d2d_get_kernel_switch(which) == on
    for which in set(range(-1, 12)) - set(declared.values()):
        assert lib.d2d_set_kernel_switch(which, 1) == _lib.ERR_INVALID
        assert lib.d2d_get_kernel_switch(which) == _lib.ERR_INVALID


def test_no_oracle_import_in_product():
    pkg = os.path.join(ROOT, "d2d-ppo_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, f"{f} references the oracle"
