"""Independent oracle of the seeded batch randomisers (schnorr_b200_batch_randomizers, include/schnorr_b200.h), written
from their definition with hashlib and Python integers; it shares no code with the device:

    s_i = int_le(SHA-512(TAG || seed || le64(i))) mod q,   TAG = b"schnorr-sig_b200/batch-randomizer/v1"
"""
import hashlib

import numpy as np

from pyref import Q

TAG = b"schnorr-sig_b200/batch-randomizer/v1"
assert len(TAG) == 36


def batch_randomizer(seed32: bytes, i: int) -> bytes:
    """Randomiser i of a 32-byte seed: 32 canonical little-endian bytes."""
    seed32 = bytes(seed32)
    assert len(seed32) == 32 and 0 <= i < 2**64
    d = hashlib.sha512(TAG + seed32 + i.to_bytes(8, "little")).digest()
    return (int.from_bytes(d, "little") % Q).to_bytes(32, "little")


def batch_randomizers(seed32: bytes, first: int, n: int) -> np.ndarray:
    """Randomisers first ... first + n - 1 as uint8[n, 32]."""
    out = np.zeros((n, 32), dtype=np.uint8)
    for k in range(n):
        out[k] = np.frombuffer(batch_randomizer(seed32, first + k), dtype=np.uint8)
    return out
