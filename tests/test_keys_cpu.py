"""The host reference of the key hash (csrc/hash.h, exported as vfb_hash_key / vfb_key_owner) restated in Python.

The GPU key tests (test_gpu_keys.py) compare every device hash with api.hash_key bit for bit, so the host function
is what pins the hash the key kernels must produce: a multilinear form over the key's zero-padded little-endian
32-bit words, each word XOR VFB_HASH_K times an odd multiplier that depends on the word index alone, then fmix64 of
the sum XOR len * VFB_HASH_L.  No GPU needed.
"""
import random

import pytest

M64 = (1 << 64) - 1
HASH_K = 0x9E3779B9
HASH_L = 0xD6E8FEB86659FD93


def fmix64(x):
    x ^= x >> 33
    x = (x * 0xFF51AFD7ED558CCD) & M64
    x ^= x >> 33
    x = (x * 0xC4CEB9FE1A85EC53) & M64
    x ^= x >> 33
    return x


def hash_mult(i):
    z = (0x9E3779B97F4A7C15 * ((i + 1) & 0xFFFFFFFF)) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    z ^= z >> 31
    return z | 1


def hash_key(key: bytes) -> int:
    padded = key + b"\0" * (-len(key) % 4)
    acc = 0
    for i in range(len(padded) // 4):
        w = int.from_bytes(padded[4 * i:4 * i + 4], "little")
        acc = (acc + (w ^ HASH_K) * hash_mult(i)) & M64
    return fmix64(acc ^ ((len(key) * HASH_L) & M64))


def key_owner(h, n_parts):
    return ((h >> 32) * n_parts) >> 32


@pytest.fixture(scope="module")
def api():
    from vfind_b200 import api, build
    build.build()
    api.load_library()
    return api


def test_hash_key_every_length_to_2100(api):
    """Every key length from 0 to 2100 bytes (the device keeps 128 multipliers in shared memory and computes the
    rest: lengths on both sides of 512 bytes), random bytes including NUL and >= 0x80, and every owner split the
    merge uses."""
    rng = random.Random(2100)
    for n in range(2101):
        key = bytes(rng.randrange(256) for _ in range(n))
        h = hash_key(key)
        assert api.hash_key(key) == h, n
        for parts in (1, 2, 7, 64, 1024):
            assert api.key_owner(h, parts) == key_owner(h, parts) < parts
    assert api.key_owner(hash_key(b"ACGT"), 0) == 0


def test_hash_key_sees_every_byte_and_the_length(api):
    """A zero byte appended changes the hash only through the length term; any one byte changed anywhere changes it."""
    rng = random.Random(7)
    for n in (1, 3, 4, 5, 79, 80, 81, 511, 512, 513, 1025):
        key = bytes(rng.randrange(256) for _ in range(n))
        h = api.hash_key(key)
        assert api.hash_key(key + b"\0") != h
        for pos in {0, n // 2, n - 1}:
            k2 = bytearray(key)
            k2[pos] ^= 1 << rng.randrange(8)
            assert api.hash_key(bytes(k2)) == hash_key(bytes(k2)) != h


def test_multipliers_are_odd_and_distinct():
    ms = [hash_mult(i) for i in range(4096)]
    assert all(m & 1 for m in ms) and len(set(ms)) == len(ms)
