"""dark_bwt_arena_bytes: the exact device bytes dark_bwt_create_ex allocates, from host arithmetic alone (no GPU here).

Up to 2^31 the values are pinned to the layout every earlier release carved; above 2^31 a context without
DARK_BWT_F_DEVICE_ONLY or DARK_BWT_F_DC_BATCH keeps one host-entry staging pair (text + BWT) instead of two."""
import pytest

from dark_b200 import _ffi, saca

D, P, O, B = _ffi.F_DEFAULT, _ffi.F_NO_ALPHABET_PACKING, _ffi.F_DEVICE_ONLY, _ffi.F_DC_BATCH
FLAG_SETS = [D, P, O, B, P | O, P | B]

# bytes the arena had before blocks above 2^31 were supported, per capacity: default, device-only, DC batch
# (alphabet packing changes no buffer)
PINNED = {
    2: (1091840, 1090816, 1094400),
    1 << 20: (48066048, 43870720, 77428736),
    1 << 28: (12026859008, 10953116160, 19543054336),
    1 << 31: (96207238656, 87617303040, 156336783360),
}


def align(b):
    return (b + 255) // 256 * 256  # every buffer of the arena starts 256-byte aligned


def pair_bytes(n):
    """One staging pair: text and BWT, N + 16 bytes each."""
    return 2 * align(n + 16)


@pytest.mark.parametrize("n", sorted(PINNED))
@pytest.mark.parametrize("flags", FLAG_SETS)
def test_pinned_layout_up_to_2_31(n, flags):
    default, device_only, dc_batch = PINNED[n]
    want = device_only if flags & O else dc_batch if flags & B else default
    assert saca.arena_bytes(n, flags) == want


@pytest.mark.parametrize("n", [(1 << 31) + 1, 5 << 29, 3 << 30, (1 << 32) - 2])
def test_one_staging_pair_above_2_31(n):
    device_only = saca.arena_bytes(n, O)
    assert saca.arena_bytes(n, D) == saca.arena_bytes(n, P) == device_only + pair_bytes(n)
    assert saca.arena_bytes(n, D) < device_only + 2 * pair_bytes(n)  # the two-pair layout of 2^31 and below
    # DC batch and device-only keep their layouts: two pairs beside the DC slots, none at all
    slots = 2 * (3 * align(4 * n + 16) + 2 * align(n + 16))  # dist, item_pos, item_dist, item_sym, item_rank, twice
    assert saca.arena_bytes(n, B) == saca.arena_bytes(n, P | B) == device_only + 2 * pair_bytes(n) + slots
    assert saca.arena_bytes(n, O) == saca.arena_bytes(n, P | O)


def test_documented_sizes():
    # include/dark_bwt.h: 96.2 GB at 2^31 (two pairs), 183.8 GB at 2^32 - 2 (one pair), 175.2 GB device-only
    assert round(saca.arena_bytes(1 << 31) / 1e9, 1) == 96.2
    assert round(saca.arena_bytes((1 << 32) - 2) / 1e9, 1) == 183.8
    assert round(saca.arena_bytes((1 << 32) - 2, O) / 1e9, 1) == 175.2


@pytest.mark.parametrize("n,flags", [(0, D), (1, D), ((1 << 32) - 1, D), (1 << 32, D), (1 << 20, O | B), (1 << 20, 8)])
def test_invalid_is_zero(n, flags):
    assert saca.arena_bytes(n, flags) == 0
