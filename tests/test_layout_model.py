"""CPU model of the shared-memory addressing used by the tensor-core build kernels (banet_b200/csrc/lm_build_tc_roles.cuh, lm_build_tc6.cu):
the 128-B swizzle with 32-B atoms (tc_utils.cuh: sw128_32b_off) and the rotated lane -> chunk walks of the b.W and R-row
loops.  Proves on the host what the kernel relies on: coverage (every element visited exactly once) and bank-conflict
freedom (each quarter-warp of a 128-bit access touches 8 distinct 16-B bank groups)."""
import itertools


def sw128_32b_off(r, c):                       # tc_utils.cuh
    return r * 128 + ((((c >> 1) ^ (r & 3)) << 5) | ((c & 1) << 4))


def test_swizzle_is_a_bijection_per_block():
    offs = {sw128_32b_off(r, c) for r in range(64) for c in range(8)}
    assert offs == set(range(0, 64 * 128, 16))                      # one 64-row x 32-float block = 8 KB, every 16-B slot once
    for r in range(64):                                             # a row stays inside its own 128 B
        assert {sw128_32b_off(r, c) // 128 for c in range(8)} == {r}


def _bank_group(off):
    return (off % 128) // 16                                        # 32 banks x 4 B = 128 B; a 16-B access spans 4 banks


def _walks(team_warp):
    """(lane, i) -> byte offset inside the 4-block basis stage, for the logical (b.W) and the physical (R rows) walk."""
    logical, physical = {}, {}
    for lane in range(32):
        r16, hf = lane & 15, lane >> 4
        nlr = team_warp * 16 + r16
        for i in range(16):
            blk, c = 2 * hf + (i >> 3), ((i & 7) + r16) & 7
            logical[(lane, i)] = (blk * 8192 + sw128_32b_off(nlr, c), blk * 32 + c * 4)     # (smem offset, W index)
            physical[(lane, i)] = hf * 16384 + nlr * 128 + (i >> 3) * 8192 + (((i & 7) + r16) & 7) * 16
    return logical, physical


def test_rotated_walks_cover_every_element_once_and_avoid_bank_conflicts():
    for w in range(4):
        logical, physical = _walks(w)
        rows = range(w * 16, w * 16 + 16)
        want = {blk * 8192 + r * 128 + s * 16 for blk in range(4) for r in rows for s in range(8)}
        assert {o for o, _ in logical.values()} == want and len(logical) == len(want)
        assert set(physical.values()) == want and len(physical) == len(want)
        for lane in range(32):                                       # the b.W walk pairs every basis column with its W entry
            cols = sorted(widx for (ln, _), (_, widx) in logical.items() if ln == lane)
            hf = lane >> 4
            assert cols == list(range(hf * 64, hf * 64 + 64, 4))
        for i, q in itertools.product(range(16), range(4)):          # a 128-bit access is served per quarter-warp
            lanes = range(8 * q, 8 * q + 8)
            assert len({_bank_group(logical[(ln, i)][0]) for ln in lanes}) == 8
            assert len({_bank_group(physical[(ln, i)]) for ln in lanes}) == 8
            assert len({(logical[(ln, i)][1] % 32) // 4 for ln in lanes}) == 8     # the W reads as well


def test_logical_column_of_a_swizzled_slot():
    """The element the kernel reads at (block, row, logical chunk c) is basis column 32*block + 4*c .. +3 of that row: the TMA
    (CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) stores logical 16-B chunk c of a row at physical slot 2*((c>>1)^(row&3)) + (c&1)."""
    for r in range(64):
        slots = [(_bank_group(sw128_32b_off(r, c))) for c in range(8)]
        assert sorted(slots) == list(range(8))
        for c in range(8):
            assert slots[c] == 2 * ((c >> 1) ^ (r & 3)) + (c & 1)
