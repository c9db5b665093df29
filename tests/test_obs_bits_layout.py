"""CPU checks of the bit-packed observation format: the header's word count, the bit order of the NumPy reference packer
the GPU tests compare against, and argument checking of the bit-packed entry points (no GPU calls are made)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from obs_bits_util import bits_words, pack_obs, unpack_obs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(6, 9), (5, 9), (6, 3), (5, 3), (6, 15), (6, 21), (6, 31), (5, 31), (6, 7)]


def test_header_macro_matches_python_helper(tmp_path):
    from primal_ppo_b200._cabi import obs_bits_words
    src = tmp_path / "w.c"
    calls = " ".join(f'printf("%d\\n", MAPF_OBS_BITS_WORDS({c}, {f}));' for c, f in SHAPES)
    src.write_text(f'#include "mapf_b200.h"\n#include <stdio.h>\nint main(void) {{ {calls} return 0; }}\n')
    exe = tmp_path / "w"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [obs_bits_words(c, f) for c, f in SHAPES] == [bits_words(c, f) for c, f in SHAPES]
    assert obs_bits_words(6, 9) == 16 and obs_bits_words(5, 9) == 13 and obs_bits_words(6, 31) == 181


@pytest.mark.parametrize("C,F", SHAPES)
def test_numpy_pack_round_trip(C, F):
    rng = np.random.default_rng(C * 100 + F)
    obs = (rng.random((3, 5, C, F, F)) < 0.3).astype(np.float32)
    words = pack_obs(obs)
    assert words.dtype == np.uint32 and words.shape == (3, 5, bits_words(C, F))
    assert np.array_equal(unpack_obs(words, C, F), obs)
    # padding bits of the last word are zero
    pad = bits_words(C, F) * 32 - C * F * F
    if pad:
        assert not np.any(words[..., -1] >> np.uint32(32 - pad))


def test_bit_order_is_lsb_first_in_reference_order():
    C, F = 6, 9
    for k in (0, 1, 31, 32, 80, 81, 485):
        obs = np.zeros((C, F, F), dtype=np.float32)
        obs.reshape(-1)[k] = 1.0
        w = pack_obs(obs)
        expect = np.zeros(bits_words(C, F), dtype=np.uint32)
        expect[k // 32] = np.uint32(1) << np.uint32(k % 32)
        assert np.array_equal(w, expect), k
    # channel c, row y, column x is bit c*F*F + y*F + x
    obs = np.zeros((C, F, F), dtype=np.float32)
    obs[2, 4, 4] = 1.0                                  # an agent's own goal at the centre of the window
    assert pack_obs(obs)[(2 * 81 + 40) // 32] == np.uint32(1) << np.uint32((2 * 81 + 40) % 32)


def test_bit_entry_points_reject_bad_arguments_without_gpu():
    from primal_ppo_b200 import _cabi
    from primal_ppo_b200.build import build
    build()
    lib = _cabi.load_library()
    E_BAD, E_NULL = -1, -2
    assert lib.mapf_observe_bits(None, None, None, None) == E_NULL
    assert lib.mapf_step_observe_bits(None, None, None, None, None, None) == E_NULL
    assert lib.mapf_unpack_obs(None, 4, 32, 6, 9, None, 4, 0, None, None) == E_NULL
    assert b"null" in lib.mapf_last_error()
    fake = ctypes.c_void_p(1 << 20)                     # never dereferenced: every check below fails before a launch
    assert lib.mapf_unpack_obs(fake, 4, 32, 6, 9, None, 4, 0, None, None) == E_NULL
    assert lib.mapf_unpack_obs(fake, 4, 32, 7, 9, None, 4, 0, fake, None) == E_BAD      # C must be 5 or 6
    assert lib.mapf_unpack_obs(fake, 4, 32, 6, 8, None, 4, 0, fake, None) == E_BAD      # F odd in 3..31
    assert lib.mapf_unpack_obs(fake, 4, 32, 6, 33, None, 4, 0, fake, None) == E_BAD
    assert lib.mapf_unpack_obs(fake, 4, 0, 6, 9, None, 4, 0, fake, None) == E_BAD       # agents >= 1
    assert lib.mapf_unpack_obs(fake, -1, 32, 6, 9, None, 4, 0, fake, None) == E_BAD     # negative rows
    assert lib.mapf_unpack_obs(fake, 4, 32, 6, 9, None, 4, 2, fake, None) == E_BAD      # out_bf16 0 or 1
    assert lib.mapf_unpack_obs(ctypes.c_void_p((1 << 20) + 2), 4, 32, 6, 9, None, 4, 0, fake, None) == E_BAD
    assert b"4-byte aligned" in lib.mapf_last_error()
    assert lib.mapf_unpack_obs(fake, 4, 32, 6, 9, None, 4, 0, ctypes.c_void_p((1 << 20) + 2), None) == E_BAD
    assert lib.mapf_unpack_obs(fake, 4, 32, 6, 9, None, 0, 0, fake, None) == 0         # nothing to do
