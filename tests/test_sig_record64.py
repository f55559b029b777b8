"""Python model of the signature construction's record word with 64-bit window positions (kc_sig_record / kc_sig_record_pos /
kc_sig_record_len, kmercamel_b200/csrc/kmerset_sig.cuh): the END position of the record's first window in bits 0..31 (low half) and
35..63 (bits 32..60), windows - 1 in bits 32..34.  Below 2^32 it must be the plain 32-bit layout {position, windows - 1} that the
kernels used before, so that inputs below 2^32 bytes keep byte-identical records."""
import random

import pytest

M64 = (1 << 64) - 1


def record(pos, length):
    """kc_sig_record"""
    return ((pos & 0xFFFFFFFF) | ((length - 1) << 32) | ((pos >> 32) << 35)) & M64


def record_pos(rec):
    """kc_sig_record_pos"""
    return (rec & 0xFFFFFFFF) | ((rec >> 35) << 32)


def record_len(rec):
    """kc_sig_record_len"""
    return ((rec >> 32) & 7) + 1


def record32(pos, length):
    """the layout before 64-bit positions: bits 0..31 position, 32..34 windows - 1"""
    return pos | ((length - 1) << 32)


@pytest.mark.parametrize("pos", [0, 1, 2**32 - 1, 2**32, 2**32 + 31, 2**33 + 5, 2**36 + 12345, 2**61 - 1])
@pytest.mark.parametrize("length", range(1, 9))
def test_record_round_trip(pos, length):
    rec = record(pos, length)
    assert 0 <= rec <= M64
    assert record_pos(rec) == pos
    assert record_len(rec) == length


def test_record_is_the_32_bit_layout_below_2_32():
    rng = random.Random(7)
    for _ in range(20000):
        pos = rng.randrange(2**32)
        length = rng.randrange(1, 9)
        assert record(pos, length) == record32(pos, length)


def test_record_order_of_positions_and_strips():
    """the resolve addresses code word pos >> 5 and reads base pos & 31 of it; both must come out of the decoded position"""
    rng = random.Random(11)
    for _ in range(20000):
        pos = rng.randrange(2**61)
        rec = record(pos, rng.randrange(1, 9))
        assert record_pos(rec) >> 5 == pos >> 5
        assert (rec & 31) == (pos & 31)  # the low half alone gives the base inside the strip



def test_scan_builds_the_high_bits_once_per_strip():
    """kc_sig_scan_kernel: record(pos0 + j, len) = 32-bit record of (pos0 mod 2^32) + j, OR the high bits of record(pos0, 1), for
    the strip start pos0 (a multiple of 32) and j < 32: a strip never crosses a multiple of 2^32"""
    rng = random.Random(5)
    for _ in range(20000):
        pos0 = rng.randrange(2**56) * 32 if rng.random() < 0.9 else 2**32 - 32 * rng.randrange(1, 4)
        j, length = rng.randrange(32), rng.randrange(1, 9)
        hi = record(pos0, 1) & ~0xFFFFFFFF & M64
        assert record(pos0 + j, length) == record32((pos0 & 0xFFFFFFFF) + j, length) | hi
