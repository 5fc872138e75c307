"""CPU tests of the batch-preparation glue (vectorised, sync-free) against the loop restatement of the
reference helpers (mm_interleaved.py:121-252).  Integer / index work: bit-exact."""
import torch

from oracle.glue import cross_attention_mask_ref, pack_mmfs_features_ref, prepare_mm_embeds_ref


def synthetic_batch(seed=0):
    g = torch.Generator().manual_seed(seed)
    BOS, IMG, SOI = 1, 32000, 32001
    L = 96
    nimg = torch.tensor([3, 0, 1, 2])
    ids = torch.randint(3, 31999, (4, L), generator=g)
    ids[:, 0] = BOS
    layout = {0: [2, 30, 60], 2: [50], 3: [1, 40]}
    for b, starts in layout.items():
        for s in starts:
            ids[b, s] = SOI
            ids[b, s + 1:s + 5] = IMG              # 4 image tokens per image in this miniature
    ids[0, 45] = BOS                                # packed-document boundary: earlier images become invisible
    ids[3, 39] = BOS
    return ids, nimg, BOS, IMG, SOI, g


def test_cross_attention_mask_matches_reference_loops():
    from mm_interleaved_b200.mm_interleaved import cross_attention_mask_from_ids
    ids, nimg, BOS, IMG, SOI, _ = synthetic_batch()
    want = cross_attention_mask_ref(ids, nimg, BOS, SOI)
    got = cross_attention_mask_from_ids(ids, int(nimg.max()), BOS, SOI, nimg)
    assert torch.equal(got, want)
    assert want[0, 44, 0] == 1 and want[0, 46, 0] == 0 and want[0, 61:, 2].all()      # the gating really bites
    # a larger static image budget only appends never-visible slots
    got5 = cross_attention_mask_from_ids(ids, 5, BOS, SOI, nimg)
    assert torch.equal(got5[..., :3], want) and got5[..., 3:].sum() == 0


def test_embed_splice_matches_reference_scatter():
    from mm_interleaved_b200.mm_interleaved import splice_image_embeds
    ids, nimg, BOS, IMG, SOI, g = synthetic_batch(1)
    C = 16
    emb = torch.randn((4, ids.shape[1], C), generator=g)
    img = torch.randn((int(nimg.sum()), 4, C), generator=g)
    soi = torch.randn((1, C), generator=g)
    want = prepare_mm_embeds_ref(emb, ids, img, soi, IMG, SOI)
    got = splice_image_embeds(emb, ids, img, soi, IMG, SOI)
    assert torch.equal(got, want)


def test_feature_packing_matches_reference_loops():
    from mm_interleaved_b200.mm_interleaved import pack_mmfs_features
    g = torch.Generator().manual_seed(2)
    nimg = torch.tensor([3, 0, 1, 2])
    feats = [torch.randn((6, 8, s, s), generator=g) for s in (16, 8, 4, 2)]
    want = pack_mmfs_features_ref(feats, [8, 4, 2], nimg)
    got = pack_mmfs_features(feats, [8, 4, 2], nimg, 3)
    assert torch.equal(got, want)


# ---- image-decoder glue (mm_interleaved.py:254-340): golden = the reference's own two methods run in the build container ----
def _imgdec_golden():
    import os

    import numpy as np
    from tests.golden.make_golden import IMGDEC_SEQ_LEN, IMGDEC_SOI, imgdec_inputs
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "imgdec_glue.npz"))
    return z, imgdec_inputs(), IMGDEC_SOI, IMGDEC_SEQ_LEN


def test_image_decoder_glue_oracle_pinned_to_reference_golden():
    from oracle.glue import context_features_for_image_decoder_ref, mmfs_features_for_image_decoder_ref
    z, (text_ids, ctx, feats, w, b, nearest_bos), soi, seq_len = _imgdec_golden()
    for tag, nb in (("a", None), ("b", nearest_bos)):
        cf, cm = context_features_for_image_decoder_ref(ctx, text_ids, soi, w, b, seq_len, nb)
        assert torch.equal(cm, torch.from_numpy(z[f"ctx_mask_{tag}"]))
        assert torch.equal(cf, torch.from_numpy(z[f"ctx_{tag}"]))                        # same ops, same order: bit-identical
        mf, mm = mmfs_features_for_image_decoder_ref(feats, text_ids, soi, nb)
        assert torch.equal(mm, torch.from_numpy(z[f"mmfs_mask_{tag}"]))
        for i, f in enumerate(mf):
            assert torch.equal(f, torch.from_numpy(z[f"mmfs_{tag}_{i}"]))


def test_image_decoder_glue_vectorised_matches_reference_golden():
    import mm_interleaved_b200.mm_interleaved as glue
    z, (text_ids, ctx, feats, w, b, nearest_bos), soi, seq_len = _imgdec_golden()
    proj = torch.nn.Linear(w.shape[1], w.shape[0])
    with torch.no_grad():
        proj.weight.copy_(w); proj.bias.copy_(b)
    n_img = feats[0].shape[0]
    for tag, nb in (("a", None), ("b", nearest_bos)):
        with torch.no_grad():
            cf, cm = glue.context_features_for_image_decoder(ctx, text_ids, soi, proj, seq_len, n_img, nb)
        want = torch.from_numpy(z[f"ctx_{tag}"])
        assert torch.equal(cm, torch.from_numpy(z[f"ctx_mask_{tag}"]))
        assert cf.shape == want.shape and (cf - want).abs().max() <= 1e-6               # same linear on the same rows (batched GEMM order)
        with torch.no_grad():   # static padding variant: longer L_max, same content under the mask
            cf2, cm2 = glue.context_features_for_image_decoder(ctx, text_ids, soi, proj, seq_len, n_img, nb, pad_to=text_ids.shape[1])
        L = want.shape[1]
        assert (cf2[:, :L] - want).abs().max() <= 1e-6 and torch.equal(cm2[:, :L], cm) and int(cm2[:, L:].sum()) == 0
        mf, mm = glue.mmfs_features_for_image_decoder(feats, text_ids, soi, nb)
        assert torch.equal(mm, torch.from_numpy(z[f"mmfs_mask_{tag}"]))
        for i, f in enumerate(mf):
            assert torch.equal(f, torch.from_numpy(z[f"mmfs_{tag}_{i}"]))


def test_sincos_1d_table_matches_the_reference_function():
    """sincos_pos_embed_1d vs utils/pos_embed.py:77-95; the reference's tables (strided rows / columns of the larger
    ones) are stored in tests/golden/sincos_1d.npz by make_golden.make_sincos."""
    import os

    import numpy as np
    import mm_interleaved_b200.mm_interleaved as glue
    from tests.golden.make_golden import SINCOS_CASES
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "sincos_1d.npz"))
    for dim, n, rows, cols in SINCOS_CASES:
        want = torch.from_numpy(z[f"d{dim}_n{n}"])
        got = glue.sincos_pos_embed_1d(dim, n)
        assert got.shape == (n, dim)
        got = got[rows, cols]
        assert got.shape == want.shape and torch.equal(got.to(want.dtype), want)


def test_soi_positions_is_nonzero_in_row_major_order():
    import mm_interleaved_b200.mm_interleaved as glue
    g = torch.Generator().manual_seed(0)
    ids = torch.randint(0, 6, (5, 33), generator=g)
    rows, cols = (ids == 3).nonzero(as_tuple=True)
    r2, c2 = glue.soi_positions(ids, 3, rows.numel())
    assert torch.equal(rows, r2) and torch.equal(cols, c2)
    r3, c3 = glue.soi_positions(ids, 3, 4)                       # a static prefix of the list
    assert torch.equal(rows[:4], r3) and torch.equal(cols[:4], c3)
