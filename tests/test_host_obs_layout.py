"""CPU checks of the host side of observations in the split-phase host call: the header's flag values, and
mapf_unpack_obs_host (the host expansion of a bit-packed slot) against the NumPy reference packer, with its argument
checks.  No GPU calls are made."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from obs_bits_util import bits_words, pack_obs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from primal_ppo_b200 import _cabi
    from primal_ppo_b200.build import build
    build()
    return _cabi.load_library()


def test_header_flags_match_python_constants(tmp_path):
    from primal_ppo_b200 import _cabi
    src = tmp_path / "f.c"
    names = ["MAPF_HOST_TRAIN_VALID", "MAPF_HOST_COMPACT", "MAPF_HOST_OBS_BF16", "MAPF_HOST_OBS_BITS", "MAPF_HOST_OBS"]
    calls = " ".join(f'printf("%d\\n", {n});' for n in names)
    src.write_text(f'#include "mapf_b200.h"\n#include <stdio.h>\nint main(void) {{ {calls} return 0; }}\n')
    exe = tmp_path / "f"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [_cabi.HOST_TRAIN_VALID, _cabi.HOST_COMPACT, _cabi.HOST_OBS_BF16, _cabi.HOST_OBS_BITS, _cabi.HOST_OBS]
    assert got == [1, 2, 4, 8, 16]


def _bits(rng, rows, N, C, F):
    obs = (rng.random((rows, N, C, F, F)) < 0.4).astype(np.float32)
    return obs, torch.from_numpy(pack_obs(obs).view(np.int32))


@pytest.mark.parametrize("C", [5, 6])
@pytest.mark.parametrize("F", [3, 9, 31])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_unpack_host_matches_numpy_packer(lib, C, F, dtype):
    from primal_ppo_b200 import unpack_observations
    rng = np.random.default_rng(C * 100 + F)
    rows, N = 7, 3
    obs, bits = _bits(rng, rows, N, C, F)
    assert tuple(bits.shape) == (rows, N, bits_words(C, F))
    want = torch.from_numpy(obs).to(dtype)
    got = unpack_observations(bits, C, F, dtype=dtype)
    assert got.dtype == dtype and not got.is_cuda and torch.equal(got, want)
    # gather through an int64 row index; out-of-range rows give zeros
    idx = torch.tensor([6, 0, -1, 3, rows, 3, -(1 << 40), 1 << 40])
    got = unpack_observations(bits, C, F, rows=idx, dtype=dtype)
    assert tuple(got.shape) == (8, N, C, F, F)
    for r, s in enumerate(idx.tolist()):
        assert torch.equal(got[r], want[s] if 0 <= s < rows else torch.zeros_like(want[0])), (r, s)
    # into a caller's buffer, whose previous contents are overwritten everywhere
    out = torch.full((rows, N, C, F, F), 7.0, dtype=dtype)
    assert unpack_observations(bits, C, F, dtype=dtype, out=out) is out and torch.equal(out, want)


def test_unpack_host_reads_only_its_rows(lib):
    """A leading-dimension slice of a larger buffer (a host slot's obs is a view into the pinned slab) is read in place,
    and only n_rows x row bytes of the output are written."""
    from primal_ppo_b200 import unpack_observations
    rng = np.random.default_rng(3)
    obs, bits = _bits(rng, 6, 4, 6, 9)
    raw = torch.full((5 * 4 * 6 * 81 + 8,), -3.0)
    out = raw[4:4 + 5 * 4 * 6 * 81].view(5, 4, 6, 9, 9)
    unpack_observations(bits[1:6], 6, 9, out=out)
    assert torch.equal(out, torch.from_numpy(obs[1:6]))
    assert bool((raw[:4] == -3.0).all() and (raw[-4:] == -3.0).all())


def test_unpack_host_rejects_bad_arguments(lib):
    E_BAD, E_NULL = -1, -2
    buf = (ctypes.c_uint32 * 4096)()
    p = ctypes.addressof(buf)
    vp = ctypes.c_void_p
    f = lib.mapf_unpack_obs_host
    assert f(None, 4, 32, 6, 9, None, 4, 0, vp(p)) == E_NULL
    assert b"null" in lib.mapf_last_error()
    assert f(vp(p), 4, 32, 6, 9, None, 4, 0, None) == E_NULL
    assert f(vp(p), 4, 32, 7, 9, None, 4, 0, vp(p)) == E_BAD        # C must be 5 or 6
    assert f(vp(p), 4, 32, 6, 8, None, 4, 0, vp(p)) == E_BAD        # F odd in 3..31
    assert f(vp(p), 4, 32, 6, 33, None, 4, 0, vp(p)) == E_BAD
    assert f(vp(p), 4, 32, 6, 1, None, 4, 0, vp(p)) == E_BAD
    assert f(vp(p), 4, 0, 6, 9, None, 4, 0, vp(p)) == E_BAD         # agents in 1..254
    assert f(vp(p), 4, 255, 6, 9, None, 4, 0, vp(p)) == E_BAD
    assert f(vp(p), -1, 32, 6, 9, None, 4, 0, vp(p)) == E_BAD       # negative row counts
    assert f(vp(p), 4, 32, 6, 9, None, -1, 0, vp(p)) == E_BAD
    assert f(vp(p), 4, 32, 6, 9, None, 4, 2, vp(p)) == E_BAD        # out_bf16 0 or 1
    assert f(vp(p + 2), 4, 32, 6, 9, None, 4, 0, vp(p)) == E_BAD    # bits 4-byte aligned
    assert b"4-byte aligned" in lib.mapf_last_error()
    assert f(vp(p), 4, 32, 6, 9, None, 4, 0, vp(p + 2)) == E_BAD    # f32 out 4-byte aligned
    assert f(vp(p), 4, 32, 6, 9, None, 4, 1, vp(p + 1)) == E_BAD    # bf16 out 2-byte aligned
    assert b"aligned" in lib.mapf_last_error()
    assert f(vp(p), 4, 32, 6, 9, None, 0, 0, vp(p)) == 0            # nothing to do


def test_unpack_host_rejects_mismatched_tensors(lib):
    from primal_ppo_b200 import unpack_observations
    bits = torch.zeros((2, 3, bits_words(6, 9)), dtype=torch.int32)
    with pytest.raises(AssertionError):
        unpack_observations(bits, 6, 7)                           # AW is not MAPF_OBS_BITS_WORDS(6, 7)
    with pytest.raises(AssertionError):
        unpack_observations(bits, 6, 9, out=torch.empty((2, 3, 6, 9, 9), dtype=torch.bfloat16))
