"""Index math of the generated-operand layouts, restated in Python and checked exhaustively (no GPU): the kernels write their
MMA operands straight into the UMMA shared-memory layouts, so a wrong offset is silent garbage and a poor thread mapping is a
bank conflict on every store.  Layout (csrc/icnn_tc3.cu, icnn_tc3_dP0_kernel): 32-bit MN-major operand tile of 16 k x 128 MN,
SWIZZLE_128B_BASE32B atoms of 4 k-rows x 128 B, LBO = 512 B between 32-wide MN blocks, SBO = 2 KB between groups of 4 k,
the 32-byte chunks of a row XOR-ed with the k-row."""
import numpy as np


def canonical_offset(k, mn):
    """Byte offset of element (k, mn) in the 16 x 128 MN-major SWIZZLE_128B_BASE32B tile."""
    return (k >> 2) * 2048 + (mn >> 5) * 512 + (k & 3) * 128 + ((((mn >> 3) & 3) ^ (k & 3)) << 5) + (mn & 7) * 4


def generator_thread(warp, lane):
    """(sample k of the stage, first of 4 consecutive MN elements, byte offset) as icnn_tc3_dP0_kernel computes them."""
    g4, hf, kr = lane >> 3, (lane >> 2) & 1, lane & 3
    ks = g4 * 4 + kr
    blk, qd = warp >> 2, warp & 3
    off = (g4 * 4 + blk) * 512 + kr * 128 + ((qd ^ kr) << 5) + hf * 16
    return ks, blk * 32 + qd * 8 + hf * 4, off


def test_dp0_generator_offsets_are_the_canonical_layout_and_cover_the_tile_once():
    seen = np.zeros(16 * 128, dtype=np.int32)
    for warp in range(16):
        for lane in range(32):
            k, mn0, off = generator_thread(warp, lane)
            assert off % 16 == 0 and off == canonical_offset(k, mn0)
            for e in range(4):                                  # the float4 store covers 4 consecutive MN elements
                assert canonical_offset(k, mn0 + e) == off + 4 * e
                seen[k * 128 + mn0 + e] += 1
    assert (seen == 1).all()                                    # 512 threads x 4 elements = the whole 16 x 128 tile, once
    offs = sorted(generator_thread(w, l)[2] for w in range(16) for l in range(32))
    assert offs == list(range(0, 8192, 16))                     # ... and the whole 8 KB of it


def test_dp0_generator_stores_are_bank_conflict_free():
    """A 16-byte store is served a quarter warp at a time: its 8 lanes must hit 8 distinct 16-byte bank groups (128 B)."""
    for warp in range(16):
        for quarter in range(4):
            groups = {(generator_thread(warp, quarter * 8 + i)[2] % 128) // 16 for i in range(8)}
            assert len(groups) == 8


def test_k_major_sw64_offsets_cover_the_tile_once():
    """K-major SWIZZLE_64B operand tiles of the forward / backward pair kernels (icnn_tc3.cu): 64-byte rows, 16-byte chunk c
    of row r at r*64 + ((c ^ ((r >> 1) & 3)) << 4); generator thread (rb, c) of icnn_tc3_fwd_kernel writes rows rb + 32 j."""
    sw64 = lambda r, c: r * 64 + ((c ^ ((r >> 1) & 3)) << 4)
    offs = sorted(sw64(r, c) for r in range(128) for c in range(4))
    assert offs == list(range(0, 128 * 64, 16))
    for rb in range(32):                                        # the kernel adds j * 2048 to the offset of (rb, c) ...
        for c in range(4):
            for j in range(4):
                assert sw64(rb + 32 * j, c) == sw64(rb, c) + j * 2048       # ... valid because 32 rows = one swizzle period
    for q in range(4):                                          # quarter warp = 2 rows x 4 chunks: 128 distinct bytes
        lanes = [(2 * q + (i >> 2), i & 3) for i in range(8)]   # t2 & 3 = chunk, (t2 >> 2) = row
        assert len({sw64(r, c) % 128 // 16 for r, c in lanes}) == 8


# ---- 16-bit MN-major operand tile of the FP16 dP0 kernel (icnn_tc3_dP0_f16_kernel): 32 k x 128 MN, SWIZZLE_128B atoms of
# 8 k-rows x 128 B (64 MN elements), LBO = 1 KB between the two atoms of a k-group, SBO = 2 KB between groups of 8 k, the
# 16-byte chunks of a row XOR-ed with the k-row (cute Swizzle<3,4,3> over ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units).
def canonical_offset_b16(k, mn):
    return (k >> 3) * 2048 + (mn >> 6) * 1024 + (k & 7) * 128 + ((((mn >> 3) & 7) ^ (k & 7)) << 4) + (mn & 7) * 2


def generator_thread_b16(warp, lane):
    """(sample k of the stage, first of 8 consecutive MN elements, byte offset) as icnn_tc3_dP0_f16_kernel computes them."""
    ncl, kg, atom, kr = lane & 7, lane >> 3, warp & 1, warp >> 1
    return kg * 8 + kr, atom * 64 + ncl * 8, kg * 2048 + atom * 1024 + kr * 128 + ((ncl ^ kr) << 4)


def test_dp0_f16_generator_offsets_are_the_canonical_layout_cover_the_tile_once_and_do_not_conflict():
    seen = np.zeros(32 * 128, dtype=np.int32)
    for warp in range(16):
        for lane in range(32):
            k, mn0, off = generator_thread_b16(warp, lane)
            assert off % 16 == 0 and off == canonical_offset_b16(k, mn0)
            for e in range(8):                                  # the 16-byte store covers 8 consecutive MN elements
                assert canonical_offset_b16(k, mn0 + e) == off + 2 * e
                seen[k * 128 + mn0 + e] += 1
        for quarter in range(4):
            assert len({(generator_thread_b16(warp, quarter * 8 + i)[2] % 128) // 16 for i in range(8)}) == 8
    assert (seen == 1).all()
    assert sorted(generator_thread_b16(w, l)[2] for w in range(16) for l in range(32)) == list(range(0, 8192, 16))
    # a K = 16 MMA step reads two consecutive 8-k groups: 4 KB from the tile start, then 4 KB more
    assert canonical_offset_b16(16, 0) == 4096 and canonical_offset_b16(8, 0) == 2048 and canonical_offset_b16(0, 64) == 1024


def test_fp16_k_major_generator_order_and_pattern_words():
    """FP16 mode of the forward / backward kernels: K-blocks of 32 (64-byte rows of fp16); the prepared table A0g holds unit
    32 kb + 8 c + e at slot 32 kb + 4 e + c (so the 4 chunk-lanes of a row read consecutive float4s), and two LeakyReLU bits
    become the packed fp16 pair (1 | 5, 1 | 5)."""
    pos = lambda c: (c & ~31) | ((c & 7) << 2) | ((c >> 3) & 3)
    assert sorted(pos(c) for c in range(256)) == list(range(256))
    for kb in range(4):
        for c in range(4):
            for e in range(8):
                assert pos(32 * kb + 8 * c + e) == 32 * kb + 4 * e + c
    half = lambda x: int(np.array([x], np.float16).view(np.uint16)[0])
    for w in range(4):
        word = 0x3C003C00 + ((w & 1) | ((w & 2) << 15)) * 0x0900
        assert word & 0xFFFF == half(5.0 if w & 1 else 1.0) and word >> 16 == half(5.0 if w & 2 else 1.0)


def test_fp16_power_of_two_scales_keep_the_operands_in_range():
    """Exponent arithmetic of the FP16 mode (icnn_tc3.cu: tensor_scale, row_scale_x1, row_scale_q1), restated on bit
    patterns: the scale is an exact power of two, scale * inverse == 1, and the scaled bound lands in the intended window."""
    bits = lambda x: int(np.array([x], np.float32).view(np.uint32)[0])
    flt = lambda b: float(np.array([b], np.uint32).view(np.float32)[0])
    clamp = lambda e, lo, hi: min(max(e, lo), hi)
    rng = np.random.default_rng(0)
    for x in np.concatenate([10.0 ** rng.uniform(-12, 12, 200), [1.0, 2.0, 0.5, 1.9999999]]).astype(np.float32):
        e = (bits(x) >> 23) & 0xFF
        et = clamp(e, 15, 253)                                  # tensor_scale: maximum -> [2^14, 2^15)
        s, inv = flt((268 - et) << 23), flt((et - 14) << 23)
        assert s * inv == 1.0 and 2.0 ** 14 <= float(x) * s < 2.0 ** 15
        ex = clamp(e, 70, 196)                                  # row_scale_x1: bound * t in [2^6, 2^7), inv = t^-2
        t, inv = flt((260 - ex) << 23), flt((2 * ex - 139) << 23)
        assert t * t * inv == 1.0 and 64.0 <= float(x) * t < 128.0
        eq = clamp(e, 30, 220)                                  # row_scale_q1 / dP0 split scale: bound * t in [2^13, 2^14)
        t, inv = flt((267 - eq) << 23), flt((eq - 13) << 23)
        assert t * inv == 1.0 and 2.0 ** 13 <= float(x) * t < 2.0 ** 14
