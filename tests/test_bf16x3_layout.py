"""Buffer sizes of the bf16x3 training path, computed from shapes (no GPU needed: the queries are host-only).

The packed image's size is read from the compile-time packed layout, the table from which the chain kernels' MMA
schedules are also derived."""

KB = 1024
TILE_DATA = 9 * 64 * KB + 32 * KB + 16 * KB + 16 * KB     # h0..h7, g | c1 | posx | posd per 128-sample tile (bf16 images)
TILE_MASKS = 8 * 4 * KB + 2 * KB                          # ReLU bit masks of h0..h7 and c1
TILE_DELTAS = 32 * KB + 9 * 64 * KB                       # delta_c1 | delta_g, delta_h7 .. delta_h0
PAD_FLOATS = 128 * 320 + 256 * 320 + 256 * 64 + 128      # padded wgrad images of color_fc.0, skip, layers_0.0 (+ fold sums)


def train_tiles(M):
    return ((M + 127) // 128 + 1) & ~1          # an even number of 128-sample tiles (pair-tiles of a CTA cluster)


def test_bf16x3_packed_image_bytes():
    from nerf_simple_b200 import _lib
    lib = _lib.load()
    slab256, slab128 = 256 * 128, 128 * 128      # bf16 operand slabs: rows x 64 K-columns x 2 B
    # forward: layers_0.0 (1 slab), 7 plain layers (4), skip (4 + posx), color_fc.0 (128 rows: 4 + posd)
    fwd = (1 + 7 * 4 + 5) * slab256 + 5 * slab128
    # delta chain: color_fc.0^T (2 K-blocks of its 128 outputs), then 8 layers of 4 K-blocks, all 256 rows
    bwd = (2 + 8 * 4) * slab256
    f32_tail = 3520 * 4
    assert lib.nb200_packed_weights_bytes(_lib.BF16X3) == 2 * fwd + f32_tail + 2 * bwd   # hi and lo of every slab


def test_bf16x3_saved_and_scratch_bytes():
    from nerf_simple_b200 import _lib
    lib = _lib.load()
    for M in (1, 128, 129, 262144):
        T = train_tiles(M)
        assert lib.nb200_mlp_saved_bytes(_lib.BF16X3, M) == T * (2 * TILE_DATA + TILE_MASKS)
        assert lib.nb200_mlp_scratch_bytes(_lib.BF16X3, M, 1) == T * 2 * TILE_DELTAS + PAD_FLOATS * 4
        assert lib.nb200_mlp_scratch_bytes(_lib.BF16X3, M, 0) == 0       # inference needs no workspace
    # 4096 rays x 64 samples: 10,512 B saved and 9,728 B of deltas per sample (2.76 GB + 2.55 GB)
    assert lib.nb200_mlp_saved_bytes(_lib.BF16X3, 262144) == 262144 * 10512
    assert lib.nb200_mlp_scratch_bytes(_lib.BF16X3, 262144, 1) == 262144 * 9728 + PAD_FLOATS * 4


def test_bf16_sizes_unchanged():
    from nerf_simple_b200 import _lib
    lib = _lib.load()
    slab256, slab128 = 256 * 128, 128 * 128
    slabs = (1 + 7 * 4 + 5) * slab256 + 5 * slab128 + (2 + 8 * 4) * slab256 + 4 * slab128 + 2 * slab256   # + folded weight
    f32_tail = (3520 + 128 * 256 + 256 * 256 + 128 * 256 + 256) * 4          # + fp32 copies for the fold / un-fold
    assert lib.nb200_packed_weights_bytes(_lib.BF16) == lib.nb200_packed_weights_bytes(_lib.BF16_LAYERWISE) == slabs + f32_tail
    for prec in (_lib.BF16, _lib.BF16_LAYERWISE):
        for M in (1, 128, 129, 262144):
            T = train_tiles(M)
            assert lib.nb200_mlp_saved_bytes(prec, M) == T * (TILE_DATA + TILE_MASKS)
            assert lib.nb200_mlp_scratch_bytes(prec, M, 1) == T * TILE_DELTAS + PAD_FLOATS * 4
