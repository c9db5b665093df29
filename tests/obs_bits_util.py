"""NumPy reference of the bit-packed observation format (include/mapf_b200.h: MAPF_OBS_BITS_WORDS): bit k of an agent's
record is obs.flatten()[k] in the [C, F, F] order, word k // 32, bit k % 32 (LSB first), padding bits 0."""
import numpy as np


def bits_words(C: int, F: int) -> int:
    return (C * F * F + 31) // 32


def pack_obs(obs: np.ndarray) -> np.ndarray:
    """[..., C, F, F] 0/1 values -> uint32 [..., AW]."""
    C, F = obs.shape[-3], obs.shape[-1]
    lead = obs.shape[:-3]
    flat = (obs.reshape(-1, C * F * F) != 0).astype(np.uint8)
    AW = bits_words(C, F)
    padded = np.zeros((flat.shape[0], AW * 32), dtype=np.uint8)
    padded[:, :C * F * F] = flat
    words = np.packbits(padded, axis=1, bitorder="little").view("<u4")
    return words.reshape(*lead, AW)


def unpack_obs(words: np.ndarray, C: int, F: int) -> np.ndarray:
    """uint32 [..., AW] -> float32 [..., C, F, F]."""
    lead = words.shape[:-1]
    bits = np.unpackbits(np.ascontiguousarray(words.astype("<u4")).view(np.uint8).reshape(-1, words.shape[-1] * 4),
                         axis=1, bitorder="little")
    return bits[:, :C * F * F].astype(np.float32).reshape(*lead, C, F, F)
