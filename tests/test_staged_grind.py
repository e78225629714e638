"""GPU: the staged proof-of-work search (zkb_grind, Winterfell's grind_query_seed) against a host brute force over the
library's host BLAKE3."""
import ctypes as C
import random

import pytest

from zk_stark_project_b200 import lib as L

pytestmark = pytest.mark.gpu


def _grind(ctx, seed, bits):
    nonce = C.c_uint64()
    ctx.check(ctx.lib.zkb_grind(ctx.handle, seed, C.c_uint32(bits), C.byref(nonce)))
    return nonce.value


def _brute_force(seed, bits):
    """smallest nonce >= 1 whose BLAKE3(seed || nonce_le64) has >= bits trailing zero bits in its first little-endian u64"""
    mask = (1 << bits) - 1
    nonce = 1
    while int.from_bytes(L.blake3_host(seed + nonce.to_bytes(8, "little"))[:8], "little") & mask:
        nonce += 1
    return nonce


@pytest.mark.parametrize("bits", [0, 1, 8, 12])
def test_grind_matches_host_brute_force(gpu_ctx, bits):
    rng = random.Random(1000 + bits)
    for _ in range(3):
        seed = bytes(rng.getrandbits(8) for _ in range(32))
        assert _grind(gpu_ctx, seed, bits) == _brute_force(seed, bits)


def test_grind_rejects_more_than_32_bits(gpu_ctx):
    with pytest.raises(L.ZkbError) as e:
        _grind(gpu_ctx, bytes(32), 33)
    assert e.value.status == -1  # ZKB_ERR_INVALID
