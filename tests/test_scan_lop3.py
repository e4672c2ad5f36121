"""The LOP3 lookup tables that mimeo_b200/csrc/seed.cu writes out for nib_merge (0x7A) and nib_rev (0xE2), evaluated bit by bit
as the `lop3.b32` instruction defines them and held against the plain expressions they replace. No GPU needed."""
import numpy as np

M32 = 0xFFFFFFFF


def lop3(a, b, c, lut):
    """bit i of the result = bit (a_i << 2 | b_i << 1 | c_i) of lut (PTX ISA, lop3: a = 0xF0, b = 0xCC, c = 0xAA)"""
    r = 0
    for i in range(32):
        k = (((a >> i) & 1) << 2) | (((b >> i) & 1) << 1) | ((c >> i) & 1)
        r |= ((lut >> k) & 1) << i
    return r


def test_lut_constants():
    assert lop3(0xF0, 0xCC, 0xAA, 0x7A) & 0xFF == 0x7A
    assert lop3(0xF0, 0xCC, 0xAA, 0xE2) & 0xFF == 0xE2


def test_nib_merge_and_nib_rev_luts_equal_the_plain_expressions():
    rng = np.random.default_rng(3)
    words = [int(x) for x in rng.integers(0, 1 << 32, 400, dtype=np.uint64)] + [0, M32, 0x88888888, 0x77777777, 0x12345678]
    for t in words:
        for q in words[:40]:
            assert lop3(t, 0x33333333, q, 0x7A) == ((t ^ q) & 0x33333333) | ((t | q) & 0xCCCCCCCC)
        x = int.from_bytes(t.to_bytes(4, 'little'), 'big')                 # __byte_perm(x, 0, 0x0123)
        got = lop3(x >> 4, 0x0F0F0F0F, (x << 4) & M32, 0xE2)
        assert got == ((x >> 4) & 0x0F0F0F0F) | ((x << 4) & 0xF0F0F0F0)
        assert got == int(''.join(reversed(f'{t:08x}')), 16)                # the eight 4-bit groups reversed
