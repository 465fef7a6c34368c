"""Launch plans of vitk_gemm_bf16 for the model's shapes (ViT-B/16@384, batch 16 → M = 9232) — host logic only.

vitk_gemm_plan runs the same planner as vitk_gemm_bf16, so these tests pin the launch that happens: the kernel
(1 = single CTA, 2 = CTA pair, 3 = CTA pair with 16 epilogue warps), the tiling and the grid.  The pair kernel deals
work items round-robin to 74 CTA pairs (148 SMs); these tests pin the decisions DESIGN.md §4 describes: 256-wide tiles
where the waves are full, mixed 256+128 tiles or 192-wide tiles for N = 768, split-K only for the weight-gradient
(accumulating) epilogue, the single-CTA kernel where the pair kernel lacks an epilogue or quantises worse."""
import pytest

import chest_x_ray_vit_b200 as pkg

ops = pkg.ops
M, D, F = 9232, 768, 3072
PAIR, PAIR16, SINGLE = 2, 3, 1


def test_wide_forward_gemms_use_256_tiles():
    fc1 = ops.gemm_plan(M, F, D, epilogue=ops.EPI_BIAS_GELUG_BF16)
    # 444 = 74 pairs × 6 tiles, on the 16-epilogue-warp instantiation
    assert fc1 == {"tile_n": 256, "split_k": 1, "n_half": 0, "work_items": 37 * 12, "kernel": PAIR16, "ctas": 148}
    # N = 2304: 333 tiles of 256 would be 4.5 waves (5 tiles on the busiest pairs); one 256-wide tile per band is
    # replaced by two 128-wide ones → 296 full + 74 half items = 4 full tiles and 1 half tile on every pair
    qkv = ops.gemm_plan(M, 3 * D, D, epilogue=ops.EPI_BIAS_BF16)
    assert qkv == {"tile_n": 256, "split_k": 1, "n_half": 2, "work_items": 37 * 10, "kernel": PAIR, "ctas": 148}


def test_fc1_variant_3_keeps_eight_epilogue_warps():
    # variant 2 forces the pair kernel, which for fc1 is the 16-warp instantiation; variant 3 is the 8-warp reference
    # with the same tiling
    fc1 = ops.gemm_plan(M, F, D, epilogue=ops.EPI_BIAS_GELUG_BF16)
    assert ops.gemm_plan(M, F, D, epilogue=ops.EPI_BIAS_GELUG_BF16, variant=2) == fc1
    assert ops.gemm_plan(M, F, D, epilogue=ops.EPI_BIAS_GELUG_BF16, variant=3) == dict(fc1, kernel=PAIR)
    # the 16-warp instantiation exists for K-major operands only
    assert ops.gemm_plan(M, F, D, epilogue=ops.EPI_BIAS_GELUG_BF16, b_mn_major=True)["kernel"] == PAIR


def test_n768_balances_the_static_schedule():
    # K-major B (forward): 192-wide tiles → 37 bands × 4 = 148 tiles = exactly two per pair
    fc2 = ops.gemm_plan(M, D, F, epilogue=ops.EPI_BIAS_RESID_F32)
    assert fc2["tile_n"] == 192 and fc2["n_half"] == 0 and fc2["work_items"] == 148
    assert fc2["kernel"] == PAIR and fc2["ctas"] == 148
    # MN-major B (dgrad): 192 is not a whole number of swizzle atoms per CTA → 2 tiles of 256 + 2 of 128 per band
    for K in (F, 3 * D, D):
        dg = ops.gemm_plan(M, D, K, epilogue=ops.EPI_STORE_BF16, b_mn_major=True)
        assert dg == {"tile_n": 256, "split_k": 1, "n_half": 2, "work_items": 148, "kernel": PAIR, "ctas": 148}, (K, dg)
    # a forced tile width switches the mixed schedule off
    assert ops.gemm_plan(M, D, F, epilogue=ops.EPI_STORE_BF16, b_mn_major=True, tile_n=256)["n_half"] == 0


def test_ragged_vit_l_data_gradients_take_the_single_cta_kernel():
    # ViT-L at batch 8: M = 4616 = 18·256 + 8.  The pair kernel's 19 bands × 4 tiles are 76 tiles on 74 pairs; the
    # single-CTA kernel's 37 bands × 4 tiles are exactly one wave on 148 SMs
    ML, DL, FL = 4616, 1024, 4096
    for K in (FL, 3 * DL, DL):
        dg = ops.gemm_plan(ML, DL, K, epilogue=ops.EPI_STORE_BF16, b_mn_major=True)
        assert dg == {"tile_n": 256, "split_k": 1, "n_half": 0, "work_items": 148, "kernel": SINGLE, "ctas": 148}, (K, dg)
        # any explicit choice keeps the pair kernel
        for pin in (dict(tile_n=256), dict(max_ctas=148), dict(variant=2)):
            assert ops.gemm_plan(ML, DL, K, epilogue=ops.EPI_STORE_BF16, b_mn_major=True, **pin)["kernel"] == PAIR, (K, pin)


def test_epilogues_without_a_pair_kernel_plan_single_cta():
    patch = ops.gemm_plan(16 * 576, D, 768, epilogue=ops.EPI_PATCH_F32, rows_in=576, rows_out=577, row_off=1)
    assert patch["kernel"] == SINGLE and patch["n_half"] == 0 and patch["ctas"] == 148
    unpatch = ops.gemm_plan(M, 768, D, epilogue=ops.EPI_UNPATCH_F32, b_mn_major=True, rows_out=577, row_off=1, ldd=384)
    assert unpatch["kernel"] == SINGLE and unpatch["n_half"] == 0
    # variant 1 forces the single-CTA kernel: 128-row bands, choose_tile_n's width
    v1 = ops.gemm_plan(M, 3 * D, D, epilogue=ops.EPI_BIAS_BF16, variant=1)
    assert v1 == {"tile_n": 192, "split_k": 1, "n_half": 0, "work_items": 73 * 12, "kernel": SINGLE, "ctas": 148}
    with pytest.raises(RuntimeError, match="CTA-pair kernel does not support"):
        ops.gemm_plan(16 * 576, D, 768, epilogue=ops.EPI_PATCH_F32, rows_in=576, rows_out=577, row_off=1, variant=2)


def test_weight_gradients_split_k_to_fill_the_pairs():
    for (m, n) in ((D, F), (F, D)):
        wg = ops.gemm_plan(m, n, M, epilogue=ops.EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
        assert wg["tile_n"] == 256 and wg["n_half"] == 0 and wg["split_k"] == 2 and wg["work_items"] == 72
        assert wg["kernel"] == PAIR and wg["ctas"] == 144
    small = ops.gemm_plan(D, D, M, epilogue=ops.EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
    assert small["split_k"] >= 4 and small["work_items"] <= 74
    # only the accumulating epilogue may split K
    assert ops.gemm_plan(D, D, M, epilogue=ops.EPI_STORE_BF16)["split_k"] == 1


def test_fewer_sms_rebalance_and_errors():
    # SMs left to a concurrent collective: the schedule is recomputed for the remaining pairs
    capped = ops.gemm_plan(M, 3 * D, D, epilogue=ops.EPI_BIAS_BF16, max_ctas=128)
    assert capped["tile_n"] in (128, 192, 256) and capped["work_items"] >= 37 * 9
    assert capped["kernel"] == PAIR and capped["ctas"] <= 128
    with pytest.raises(RuntimeError):
        ops.gemm_plan(M, 100, D, epilogue=ops.EPI_STORE_BF16)           # N must be a multiple of 128
