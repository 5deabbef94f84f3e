"""-m gpu: cross-modal retrieval (MultiModalLitModel.evaluate_retrieval, ops.retrieval_f32, cvcl_rank_topk_f32).
Top-k, ranks and gathered scores equal the literal sort of the full score matrix built by the existing fp32 ops bit for
bit, for every block size; against fp64 they differ only at fp32 near-ties."""
import argparse
import math

import numpy as np
import pytest
import torch

from _retrieval import assert_within_near_ties, scores_fp64, sorted_reference
from _util import O, S_DEFAULT, case_inputs, t

pytestmark = pytest.mark.gpu
DEV = "cuda"
V = 2350


@pytest.fixture(scope="module")
def cv():
    import multimodal_baby_b200 as m
    m._cabi.load()
    return m


def _lit(cv, etype, sim="max", E=512, normalize=True, seed=0):
    args = argparse.Namespace(embedding_type=etype, embedding_dim=E, normalize_features=normalize,
                              fix_temperature=True, temperature=0.07, text_encoder="embedding", sim=sim)
    vocab = {"<pad>": 0, "<unk>": 1, "<sos>": 2, "<eos>": 3, **{"w%d" % i: i for i in range(4, V)}}
    lit = cv.MultiModalLitModel(cv.VisionEncoder(args, trunk="pooled"), cv.TextEncoder(vocab, 2048, args), args,
                                vocab=vocab)
    rng = np.random.RandomState(seed)
    W, b, table = O.synth_weights(rng, E, 2048, V)
    with torch.no_grad():
        if etype == "flat":
            lit.model.image_embed.model.fc.weight.copy_(t(W)); lit.model.image_embed.model.fc.bias.copy_(t(b))
        else:
            conv = lit.model.image_embed.model[-1]
            conv.weight.copy_(t(W)[:, :, None, None]); conv.bias.copy_(t(b))
        lit.model.text_embed.embedding.weight.copy_(t(table))
    return lit.to(DEV).eval(), (t(W), t(b), t(table))


def _rows_per_block(rows, n_keys):
    return 1 << 30 if rows is None else rows * 4 * n_keys


def _check_exact(res, s_i2t, s_t2i, fg, tg, k, scale, recall_at=(1, 5, 10)):
    """res against sorted_reference on the full fp32 score matrices (logits = scale * gathered score)."""
    for name, s, qg, kg in (("image_to_text", s_i2t, fg, tg), ("text_to_image", s_t2i, tg, fg)):
        d = res[name]
        topk, rank = sorted_reference(s, qg, kg, k)
        assert d["topk"].dtype == torch.int32 and d["rank"].dtype == torch.int32
        assert np.array_equal(d["topk"].cpu().numpy(), topk), name
        assert np.array_equal(d["rank"].cpu().numpy(), rank), name
        vals = torch.gather(s, 1, d["topk"].long())
        torch.testing.assert_close(d["logits"], vals if scale is None else vals * scale, rtol=0, atol=0,
                                   equal_nan=True)
        # rank < k iff a positive is in the top-k
        if qg is None:
            in_topk = (topk == np.arange(len(rank))[:, None]).any(axis=1)
        else:
            in_topk = (kg.cpu().numpy()[topk] == qg.cpu().numpy()[:, None]).any(axis=1)
        assert np.array_equal((rank >= 0) & (rank < k), in_topk)
        r = rank[rank >= 0] + 1
        assert d["n_queries"] == len(r)
        if len(r):
            assert d["median_rank"] == float(np.sort(r)[(len(r) - 1) // 2])
            assert d["mean_rank"] == pytest.approx(r.mean(), rel=1e-12)
            for K in recall_at:
                assert d["recall"][K] == pytest.approx((r <= K).mean(), rel=1e-12)
        else:
            assert np.isnan(d["median_rank"]) and np.isnan(d["mean_rank"])


def _same(a, b):
    for name in ("image_to_text", "text_to_image"):
        for f in ("topk", "rank"):
            assert torch.equal(a[name][f], b[name][f])
        torch.testing.assert_close(a[name]["logits"], b[name]["logits"], rtol=0, atol=0, equal_nan=True)
        assert a[name]["recall"] == b[name]["recall"] and a[name]["n_queries"] == b[name]["n_queries"]


# ------------------------------------------------------------------------------------------------ the kernel
@pytest.mark.parametrize("k", [1, 10, 64])
def test_rank_topk_kernel_on_crafted_rows(cv, k):
    """rows that rise along the key index (the candidate list is cut at every tile), ties, NaNs and -0 / +0,
    pair and group mode, a block that starts at a query offset."""
    g = torch.Generator(device=DEV).manual_seed(k)
    M, N = 48, 5000
    s = torch.randn((M, N), generator=g, device=DEV)
    s[0] = torch.arange(N, device=DEV, dtype=torch.float32)           # ascending
    s[1] = -torch.arange(N, device=DEV, dtype=torch.float32)          # descending
    s[2] = 1.0                                                         # all tied
    s[3] = float("nan")                                                # all NaN
    s[4:20, ::7] = s[4:20, 3:4]                                        # many ties with key 3
    s[5:9, 4000] = float("nan")
    s[6, 17] = float("nan")
    s[10:14, ::2] = 0.0
    s[10:14, 1::2] = -0.0
    s = torch.round(s * 8) / 8                                         # coarse values: ties everywhere
    qg = torch.randint(0, 9, (M,), generator=g, device=DEV)
    kg = torch.randint(0, 8, (N,), generator=g, device=DEV)           # group 8: no positive
    for q0, groups in ((0, None), (0, (qg, kg)), (1000, None)):
        topk = torch.empty((M, k), dtype=torch.int32, device=DEV)
        val = torch.empty((M, k), dtype=torch.float32, device=DEV)
        rank = torch.empty((M,), dtype=torch.int32, device=DEV)
        qgp = cv.ops._p(groups[0]) if groups else None
        kgp = cv.ops._p(groups[1]) if groups else None
        cv._cabi.call("cvcl_rank_topk_f32", cv.ops._p(s), N, M, N, q0, qgp, kgp, k, cv.ops._p(topk), cv.ops._p(val),
                      cv.ops._p(rank), cv.ops._stream())
        if groups:
            ref_topk, ref_rank = sorted_reference(s, qg, kg, k)
        else:
            full = torch.full((q0 + M, N), 0.0, device=DEV)
            full[q0:] = s
            ref_topk, ref_rank = sorted_reference(full, None, None, k)
            ref_topk, ref_rank = ref_topk[q0:], ref_rank[q0:]
        assert np.array_equal(topk.cpu().numpy(), ref_topk)
        assert np.array_equal(rank.cpu().numpy(), ref_rank)
        torch.testing.assert_close(val, torch.gather(s, 1, topk.long()), rtol=0, atol=0, equal_nan=True)
    assert topk[0].tolist() == list(range(N - 1, N - 1 - k, -1)) and topk[3].tolist() == list(range(k))


# ------------------------------------------------------------------------------------------------ exact, flat
@pytest.fixture(scope="module")
def flat_feats():
    """3000 frames and texts, E = 512; text i near frame i; duplicate and scaled-copy rows across block edges."""
    g = torch.Generator(device=DEV).manual_seed(11)
    img = torch.randn((3000, 512), generator=g, device=DEV)
    txt = img + 2.0 * torch.randn((3000, 512), generator=g, device=DEV)
    for a, b in ((6, 7), (998, 999), (1500, 2999)):
        img[b] = img[a]; txt[b] = 2.0 * txt[a]
    return img, txt


@pytest.mark.parametrize("normalize", [True, False])
def test_flat_exact_against_existing_ops(cv, flat_feats, normalize):
    img, txt = flat_feats
    i = cv.ops.normalize_rows_f32(img) if normalize else img
    tt = cv.ops.normalize_rows_f32(txt) if normalize else txt
    s_i2t, s_t2i = cv.ops.linear_f32(i, tt, None), cv.ops.linear_f32(tt, i, None)
    assert torch.equal(s_t2i, s_i2t.t())                              # one fmaf per k in ascending k, both ways
    scale = math.exp(S_DEFAULT)
    res = cv.ops.retrieval_f32(img, txt, None, "flat", normalize, S_DEFAULT)
    _check_exact(res, s_i2t, s_t2i, None, None, 10, scale)
    assert res["image_to_text"]["recall"][10] > 0.5                  # text i is near frame i
    for rows in (1, 7, 999):
        _same(cv.ops.retrieval_f32(img, txt, None, "flat", normalize, S_DEFAULT,
                                   block_bytes=_rows_per_block(rows, 3000)), res)
    _same(cv.ops.retrieval_f32(img, txt, None, "flat", normalize, S_DEFAULT), res)      # replay
    # group mode, k = 64
    g = torch.Generator(device=DEV).manual_seed(12)
    fg = torch.randint(0, 300, (3000,), generator=g, device=DEV)
    tg = torch.randint(0, 300, (3000,), generator=g, device=DEV)
    res = cv.ops.retrieval_f32(img, txt, None, "flat", normalize, S_DEFAULT, fg, tg, k=64, recall_at=(1, 64))
    _check_exact(res, s_i2t, s_t2i, fg, tg, 64, scale, (1, 64))
    _same(cv.ops.retrieval_f32(img, txt, None, "flat", normalize, S_DEFAULT, fg, tg, k=64, recall_at=(1, 64),
                               block_bytes=_rows_per_block(7, 3000)), res)


# ------------------------------------------------------------------------------------------------ exact, spatial
@pytest.fixture(scope="module")
def maps300():
    g = torch.Generator(device=DEV).manual_seed(21)
    return torch.randn((300, 2048, 7, 7), generator=g, device=DEV).relu_()


def _texts(n, L, seed):
    rng = np.random.RandomState(seed)
    lens = rng.randint(1, L + 1, size=n).astype(np.int64)
    lens[:3] = [1, L, (L + 1) // 2]
    ids = np.zeros((n, L), np.int64)
    for c in range(n):
        ids[c, :lens[c]] = rng.randint(4, V, size=lens[c])
    return t(ids, DEV), t(lens, DEV)


@pytest.mark.parametrize("from_trunk", [True, False])
@pytest.mark.parametrize("L", [1, 3, 25])
@pytest.mark.parametrize("sim", ["max", "mean"])
def test_spatial_exact_against_existing_ops(cv, maps300, sim, L, from_trunk):
    lit, _ = _lit(cv, "spatial", sim, seed=L)
    ids, lens = _texts(300, L, L)
    heads = lit._spatial_head_outputs(maps300, (), True, "test")                 # [300, 49, E]
    frames = maps300 if from_trunk else heads.view(300, 7, 7, 512).permute(0, 3, 1, 2)
    txt = lit._spatial_text(ids, lens, 49)
    rows = cv.ops._location_rows(heads, True)
    s = cv.ops._scalar(lit.model.logit_neg_log_temperature)
    if sim == "max":
        s_i2t = cv.ops._spatial_max_scores(rows, txt, lens, None, 0, s)
        s_t2i, scale = s_i2t.t(), None
    else:
        pooled = cv.ops.spatial_pool(rows)
        s_i2t, s_t2i = cv.ops.linear_f32(pooled, txt, None), cv.ops.linear_f32(txt, pooled, None)
        assert torch.equal(s_t2i, s_i2t.t())
        scale = math.exp(s)
    res = lit.evaluate_retrieval(frames, ids, lens, from_trunk_boundary=from_trunk)
    _check_exact(res, s_i2t, s_t2i, None, None, 10, scale)
    for rows_per in (1, 7, 999):
        _same(lit.evaluate_retrieval(frames, ids, lens, from_trunk_boundary=from_trunk,
                                     block_bytes=_rows_per_block(rows_per, 300)), res)
    _same(lit.evaluate_retrieval(frames, ids, lens, from_trunk_boundary=from_trunk), res)   # replay


# ------------------------------------------------------------------------------------------------ ties, NaN, no positive
@pytest.mark.parametrize("sim", ["flat", "mean", "max"])
def test_ties_nans_and_queries_without_positive(cv, sim):
    g = torch.Generator(device=DEV).manual_seed(31)
    n, E = 200, 64
    if sim == "flat":
        img = torch.randn((n, E), generator=g, device=DEV)
        txt = torch.randn((n, E), generator=g, device=DEV)
        lens = None
    else:
        img = torch.randn((n, 49, E), generator=g, device=DEV)
        txt = torch.randn((n, 3, E) if sim == "max" else (n, E), generator=g, device=DEV)
        lens = torch.full((n,), 3, dtype=torch.int64, device=DEV)
    for a, b in ((6, 7), (13, 14), (100, 199)):                      # duplicates and scaled copies across blocks
        img[b] = 2.0 * img[a]; txt[b] = txt[a]
    img[50] = float("nan")                                             # a NaN frame: first for every text
    fg = torch.arange(n, device=DEV) % 17
    tg = torch.arange(n, device=DEV) % 17
    fg[:10] = 50; tg[190:] = 40                                        # no text of group 50, no frame of group 40
    if sim == "max":
        rows = cv.ops._location_rows(img, True)
        s_i2t = cv.ops._spatial_max_scores(rows, txt, lens, None, 0, 0.0)
        s_t2i, scale = s_i2t.t(), None
    else:
        i = cv.ops.normalize_rows_f32(img) if sim == "flat" else cv.ops.spatial_pool(cv.ops._location_rows(img, True))
        tt = cv.ops.normalize_rows_f32(txt) if sim == "flat" else txt
        s_i2t, s_t2i, scale = cv.ops.linear_f32(i, tt, None), cv.ops.linear_f32(tt, i, None), 1.0
    for groups in ((None, None), (fg, tg)):
        for rows_per in (None, 7):
            res = cv.ops.retrieval_f32(img, txt, lens, sim, True, 0.0, *groups, k=16,
                                       block_bytes=_rows_per_block(rows_per, n))
            _check_exact(res, s_i2t, s_t2i, *groups, 16, scale)
            assert res["text_to_image"]["topk"][:, 0].eq(50).all()
            assert res["image_to_text"]["topk"][50].tolist() == list(range(16))
    assert (res["image_to_text"]["rank"][:10] == -1).all() and res["image_to_text"]["n_queries"] == n - 10
    assert (res["text_to_image"]["rank"][190:] == -1).all() and res["text_to_image"]["n_queries"] == 190


# ------------------------------------------------------------------------------------------------ fp64
@pytest.mark.parametrize("sim", ["flat", "mean", "max"])
def test_against_fp64_up_to_near_ties(cv, sim):
    n = 1000 if sim == "flat" else 300
    etype = "flat" if sim == "flat" else "spatial"
    lit, (W, b, table) = _lit(cv, etype, sim, seed=41)
    inp = case_inputs(42, n, 512, etype)
    f, ids, lens = t(inp["f"], DEV), t(inp["ids"], DEV), t(inp["lens"], DEV)
    ids[n // 2:] = ids[: n - n // 2]; lens[n // 2:] = lens[: n - n // 2]          # repeated utterances
    res = lit.evaluate_retrieval(f, ids, lens, k=20)
    s64 = scores_fp64(sim, f, W.to(DEV), b.to(DEV), ids, lens, table.to(DEV))
    for name, s in (("image_to_text", s64), ("text_to_image", s64.t())):
        assert_within_near_ties(res[name]["topk"], res[name]["rank"], s, None, None, "%s %s" % (sim, name))


# ------------------------------------------------------------------------------------------------ existing API
@pytest.mark.parametrize("sim", ["flat", "mean", "max"])
def test_category_retrieval_matches_classify_frames(cv, sim):
    """the 22 category labels as the texts, each frame's category as its group: the top text is classify_frames'
    prediction and its logit the classify_frames logit, bit for bit."""
    etype = "flat" if sim == "flat" else "spatial"
    lit, _ = _lit(cv, etype, sim, seed=51)
    inp = case_inputs(52, 120, 512, etype)
    f = t(inp["f"], DEV)
    ids, lens = t(inp["ids"][:22], DEV), t(inp["lens"][:22], DEV)
    pred, logits = lit.classify_frames(f, ids, lens)
    cat = torch.randint(0, 22, (120,), generator=torch.Generator(device=DEV).manual_seed(53), device=DEV)
    res = lit.evaluate_retrieval(f, ids, lens, frame_group=cat, text_group=torch.arange(22, device=DEV), k=5)
    i2t = res["image_to_text"]
    assert torch.equal(i2t["topk"][:, 0], pred)
    assert torch.equal(i2t["logits"][:, 0], logits.gather(1, pred.long()[:, None])[:, 0])
    assert torch.equal(i2t["logits"], logits.gather(1, i2t["topk"].long()))
    acc = float((pred.long() == cat).double().mean())
    assert i2t["recall"][1] == pytest.approx(acc, rel=1e-12) and i2t["n_queries"] == 120
    assert res["text_to_image"]["n_queries"] == int(torch.unique(cat).numel())


@pytest.mark.parametrize("sim", ["flat", "max"])
def test_grouped_repeated_utterances_rank_no_worse_than_pairs(cv, sim):
    etype = "flat" if sim == "flat" else "spatial"
    lit, _ = _lit(cv, etype, sim, seed=61)
    inp = case_inputs(62, 240, 512, etype)
    f, ids, lens = t(inp["f"], DEV), t(inp["ids"], DEV), t(inp["lens"], DEV)
    rep = torch.arange(240, device=DEV) % 60                          # 60 utterances, each said four times
    ids, lens = ids[rep], lens[rep]
    _, grp = torch.unique(ids, dim=0, return_inverse=True)
    pair = lit.evaluate_retrieval(f, ids, lens, k=10)
    group = lit.evaluate_retrieval(f, ids, lens, frame_group=grp, text_group=grp, k=10)
    for name in ("image_to_text", "text_to_image"):
        assert (group[name]["rank"] <= pair[name]["rank"]).all()
        assert group[name]["recall"][1] >= pair[name]["recall"][1]
    assert (group["image_to_text"]["rank"] < pair["image_to_text"]["rank"]).any()   # pair mode undercounts hits
