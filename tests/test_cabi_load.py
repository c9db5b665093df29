"""CPU-side checks of the boundary: the CUDA library builds, loads and exports every symbol include/mapf_b200.h
declares.  No compute calls are made (there is no GPU here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib_path():
    from primal_ppo_b200.build import build
    return build()


def test_header_symbols_exported(lib_path):
    hdr = open(os.path.join(ROOT, "include", "mapf_b200.h")).read()
    body = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(mapf_[a-z_0-9]+)\s*\(", body))
    assert {"mapf_create", "mapf_step", "mapf_observe", "mapf_bfs", "mapf_gae"} <= declared
    lib = ctypes.CDLL(lib_path)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in mapf_b200.h but not exported"
    lib.mapf_abi_version.restype = ctypes.c_int
    m = re.search(r"#define MAPF_B200_ABI_VERSION (\d+)", hdr)
    assert lib.mapf_abi_version() == int(m.group(1))


def test_python_binding_lists_every_symbol(lib_path):
    from primal_ppo_b200 import _cabi
    hdr = open(os.path.join(ROOT, "include", "mapf_b200.h")).read()
    body = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(mapf_[a-z_0-9]+)\s*\(", body))
    assert declared == set(_cabi.EXPORTED)
    lib = _cabi.load_library()
    assert lib.mapf_abi_version() == _cabi.ABI_VERSION == 2


def test_config_struct_layout_matches_header():
    from primal_ppo_b200 import _cabi
    assert ctypes.sizeof(_cabi.MapfConfig) == 12 * 4 + 8 + 4 * 4
    assert _cabi.MapfConfig.seed.offset == 48
    assert _cabi.MapfConfig.goal_sampling.offset == 64
    assert ctypes.sizeof(_cabi.MapfScenario) == 9 * 8
    assert ctypes.sizeof(_cabi.MapfStepOut) == 10 * 8
    assert ctypes.sizeof(_cabi.MapfHostLayout) == 10 * 8


def test_null_arguments_are_rejected_without_gpu(lib_path):
    from primal_ppo_b200 import _cabi
    lib = _cabi.load_library()
    assert lib.mapf_create(None, None) == -2
    assert b"null" in lib.mapf_last_error()
    assert lib.mapf_step(None, None, None, None) == -2
    assert lib.mapf_gae(None, None, None, None, 0.95, 0.95, 4, 4, None, None, None) == -2


def test_env_refuses_to_run_without_cuda(monkeypatch):
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)      # also on a machine that has a GPU
    from primal_ppo_b200 import BatchedMapfGym, random_scenario
    from primal_ppo_b200._cabi import MapfError
    with pytest.raises(MapfError):
        BatchedMapfGym(random_scenario(2, 8, 8, 2, seed=0))


def test_header_is_plain_c_and_links(lib_path, tmp_path):
    """include/mapf_b200.h compiles as C99 (no C++, no torch types) and a C program links against the library."""
    import subprocess
    src = tmp_path / "t.c"
    src.write_text('#include "mapf_b200.h"\n#include <stdio.h>\nint main(void) { MapfConfig c; MapfScenario s; MapfStepOut o; '
                   'MapfGenConfig g; MapfHostLayout l; (void)c; (void)s; (void)o; (void)g; (void)l; '
                   'printf("%d %d %d %d %d\\n", mapf_abi_version(), mapf_create(0, 0), (int)sizeof(MapfConfig), (int)sizeof(MapfStepOut), '
                   '(int)sizeof(MapfHostLayout)); return 0; }\n')
    exe = tmp_path / "t"
    libdir = os.path.dirname(lib_path)
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                    "-o", str(exe), "-L", libdir, "-l:" + os.path.basename(lib_path), "-Wl,-rpath," + libdir], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    from primal_ppo_b200 import _cabi
    assert out == ["2", "-2", str(ctypes.sizeof(_cabi.MapfConfig)), str(ctypes.sizeof(_cabi.MapfStepOut)),
                   str(ctypes.sizeof(_cabi.MapfHostLayout))]


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """No silent fallback: without the built .so every entry into the product raises."""
    from primal_ppo_b200 import _cabi
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(_cabi, "LIB_PATH", str(tmp_path / "libmapf_b200.so"))
    with pytest.raises(_cabi.MapfError, match="no CPU fallback|missing"):
        _cabi.load_library()


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under primal_ppo_b200/ may import it."""
    pkg = os.path.join(ROOT, "primal_ppo_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), os.path.join(dirpath, f)
