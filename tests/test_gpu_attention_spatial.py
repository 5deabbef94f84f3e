"""-m gpu: text-to-location attention maps of spatial-embedding models (ops.spatial_attention_f32,
MultiModalModel.spatial_attention_maps) against the fp64 reference of tests/_spatial_attention.py, and bit for bit
against the spatial "max" scores the evaluation path computes."""
import argparse

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from _spatial_attention import spatial_attention_maps
from _spatial_eval import match_fp64

pytestmark = pytest.mark.gpu
DEV = "cuda"
V = 2350


@pytest.fixture(scope="module")
def cv():
    import multimodal_baby_b200 as m
    m._cabi.load()
    return m


def _case(seed, M, HW, E, L, with_index):
    """M images of HW locations and C label rows with ragged lengths (1, L and random ones; with an index also an
    empty label, and one image whose index is out of range)."""
    rng = np.random.RandomState(seed)
    u = torch.from_numpy(rng.standard_normal((M, E, HW, 1)).astype(np.float32))
    u[0, :, HW - 1] = u[0, :, 0]                             # an exact tie between two locations of image 0
    table = torch.from_numpy(rng.standard_normal((V, E)).astype(np.float32))
    table[0] = 0
    C = M + 2 if with_index else M
    lens = rng.randint(1, L + 1, size=C)
    lens[0], lens[1] = L, 1
    if with_index:
        lens[2] = 0
    ids = np.zeros((C, L), np.int64)
    for c in range(C):
        ids[c, :lens[c]] = rng.randint(4, V, size=lens[c])
    index = torch.from_numpy(rng.randint(0, C, size=M).astype(np.int32)) if with_index else None
    if with_index:
        index[:3] = torch.tensor([0, 2, 1], dtype=torch.int32)
        index[3] = C                                       # out of range: NaN maps
    return u, table, torch.from_numpy(ids), torch.from_numpy(lens.astype(np.int64)), index


def _nan_equal(a, b):
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a[~na], b[~nb])


@pytest.mark.parametrize("with_index", [True, False])
@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("HW,E,L", [(49, 512, 3), (49, 512, 25), (49, 64, 1), (1, 512, 4), (64, 128, 77)])
def test_maps_vs_fp64_and_the_max_scores_bit_for_bit(cv, HW, E, L, normalize, with_index):
    M = 24
    u, table, ids, lens, index = _case(HW * 7 + E + L + 3 * normalize + with_index, M, HW, E, L, with_index)
    d_lens = lens.to(DEV)
    tok, _ = cv.ops.text_features_spatial(ids.to(DEV), d_lens, table.to(DEV), normalize)
    img = u.reshape(M, E, HW).permute(0, 2, 1).contiguous().to(DEV)            # NHWC rows [M, HW, E]
    d_index = None if index is None else index.to(DEV)
    maps, utt, arg = cv.ops.spatial_attention_f32(img, tok, d_lens, d_index, normalize)
    assert maps.shape == (M, L, HW) and utt.shape == (M, HW) and arg.shape == (M, L) and arg.dtype == torch.int32
    maps, utt, arg = maps.cpu(), utt.cpu(), arg.cpu()

    pair = torch.arange(M) if index is None else index.long()
    ok = pair < ids.shape[0]                                                   # images with a label
    bad = torch.nonzero(~ok).flatten()
    assert bool(torch.isnan(maps[bad]).all() and torch.isnan(utt[bad]).all() and (arg[bad] == -1).all())
    pair, rows = pair[ok], torch.nonzero(ok).flatten()
    n = lens[pair]
    T64, U64 = spatial_attention_maps(u[rows], ids[pair], n, table, normalize)
    T64, U64 = T64.reshape(len(rows), L, HW), U64.reshape(len(rows), HW)
    T, U, A = maps[rows], utt[rows], arg[rows]
    live = torch.arange(L)[None, :] < n[:, None]
    # pads: exactly 0, arg-max -1; an empty label gives NaN utterance maps (0 / 0, as the reference divides)
    assert bool((T[~live] == 0).all()) and bool((A[~live] == -1).all())
    empty = n == 0
    assert bool(torch.isnan(U[empty]).all())
    # token and utterance maps within 2e-6 of each image's largest sum_e |x_e t_e|, the magnitude an fp32 dot's
    # rounding scales with.  It is the largest |map| up to a small factor when there are many locations; with one
    # location and one live token the map can be a cancellation far below it (fp32 torch.einsum then misses
    # 2e-6 * max|map| by 10x).
    A64, _ = spatial_attention_maps(u[rows].abs(), ids[pair], n, table.abs(), normalize)
    for k in torch.nonzero(~empty).flatten().tolist():
        scale = float(A64[k].max())
        assert float((T[k].double() - T64[k]).abs().max()) <= 2e-6 * scale, k
        assert float((U[k].double() - U64[k]).abs().max()) <= 2e-6 * scale, k

    # the loss path's "max" scores, trial mode at log_scale 0: the same dots, bit for bit
    rows_n = cv.ops._location_rows(img, normalize)
    scores = cv.ops._spatial_max_scores(rows_n, tok, d_lens, d_index, 1, 0.0).cpu()
    assert bool(torch.isnan(scores[bad]).all())
    tmax = torch.where(live, T.amax(dim=-1), torch.zeros(()))
    acc = torch.zeros(len(rows), dtype=torch.float32)
    for l in range(L):                                                         # fp32, position order
        acc = torch.where(live[:, l], acc + tmax[:, l], acc)
    assert _nan_equal(acc / n.float(), scores[rows])
    # every arg-max is the first location holding its token's maximum
    first = torch.argmax(T, dim=-1).to(torch.int32)
    assert torch.equal(torch.where(live, first, torch.full_like(first, -1)), A)
    assert HW == 1 or int(A[0, 0]) < HW - 1                                    # the tie goes to the lower location

    # the mean identity: the mean over the locations of U is the sim="mean" match
    ok_mean = ~empty
    ref = match_fp64(u[rows].reshape(-1, E, HW, 1), ids, lens, table, "mean", normalize)[torch.arange(len(rows)), pair]
    got = U.double().mean(dim=-1)
    assert float((got[ok_mean] - ref[ok_mean]).abs().max()) <= 2e-6 * float(ref[ok_mean].abs().max())

    # utterance maps only
    e1, utt2, e2 = cv.ops.spatial_attention_f32(img, tok, d_lens, d_index, normalize, want_tokens=False)
    assert e1.numel() == 0 and e2.numel() == 0 and _nan_equal(utt2.cpu(), utt)


def _spatial_model(cv, E=512, normalize=True, seed=11):
    args = argparse.Namespace(embedding_type="spatial", embedding_dim=E, normalize_features=normalize,
                              fix_temperature=True, temperature=0.07, text_encoder="embedding", sim="max")
    vocab = {"<pad>": 0, "<unk>": 1, "<sos>": 2, "<eos>": 3, **{"w%d" % i: i for i in range(4, V)}}
    lit = cv.MultiModalLitModel(cv.VisionEncoder(args, trunk="pooled"), cv.TextEncoder(vocab, 2048, args), args,
                                vocab=vocab)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        conv = lit.model.image_embed.model[-1]
        conv.weight.copy_(torch.randn(E, 2048, 1, 1, generator=g) / 45)
        conv.bias.copy_(torch.randn(E, generator=g) / 45)
        tab = torch.randn(V, E, generator=g)
        tab[0] = 0
        lit.model.text_embed.embedding.weight.copy_(tab)
    return lit.to(DEV).eval()


def test_model_maps_equal_the_op_on_the_fp32_head_and_resize_like_interpolate(cv):
    lit = _spatial_model(cv)
    m = lit.model
    N, C, L = 6, 4, 25
    g = torch.Generator().manual_seed(12)
    fmap = torch.randn(N, 2048, 7, 7, generator=g).relu_().to(DEV)
    ids = torch.zeros((C, L), dtype=torch.int64)
    lens = torch.tensor([3, 1, 25, 7])
    for c in range(C):
        ids[c, :lens[c]] = torch.randint(4, V, (int(lens[c]),), generator=g)
    ids, lens = ids.to(DEV), lens.to(DEV)
    index = torch.tensor([0, 1, 2, 3, 2, 0], dtype=torch.int32, device=DEV)

    utt, maps, arg = m.spatial_attention_maps(fmap, ids, lens, index)
    assert utt.shape == (N, 1, 7, 7) and maps.shape == (N, L, 7, 7) and arg.shape == (N, L)
    w, b = m._head()
    rows = cv.ops.conv1x1_f32(fmap, w, b).view(N, 49, -1)
    tok, _ = cv.ops.text_features_spatial(ids, lens, m.text_embed.embedding.weight, True)
    maps_op, utt_op, arg_op = cv.ops.spatial_attention_f32(rows, tok, lens, index, True)
    assert torch.equal(maps.reshape(N, L, 49), maps_op) and torch.equal(utt.reshape(N, 49), utt_op)
    assert torch.equal(arg, arg_op)

    # resized utterance maps: CPU F.interpolate of the kernel's own 7x7 maps within 2e-5 of the largest value
    big, maps2, arg2 = lit.attention_maps(fmap, ids, lens, index, out_size=(224, 224))
    assert big.shape == (N, 1, 224, 224) and torch.equal(maps2, maps) and torch.equal(arg2, arg)
    ref = F.interpolate(utt.cpu(), size=(224, 224), mode="bicubic", align_corners=False)
    assert float((big.cpu() - ref).abs().max()) <= 2e-5 * float(ref.abs().max())
    assert lit.attention_maps(fmap, ids, lens, index, out_size=112)[0].shape == (N, 1, 112, 112)


def test_graph_replay_is_bit_identical(cv):
    M, HW, E, L = 40, 49, 512, 25
    u, table, ids, lens, index = _case(99, M, HW, E, L, True)
    d_lens, d_index = lens.to(DEV), index.to(DEV)
    tok, _ = cv.ops.text_features_spatial(ids.to(DEV), d_lens, table.to(DEV), True)
    img = u.reshape(M, E, HW).permute(0, 2, 1).contiguous().to(DEV)
    eager = cv.ops.spatial_attention_f32(img, tok, d_lens, d_index, True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        cv.ops.spatial_attention_f32(img, tok, d_lens, d_index, True)        # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = cv.ops.spatial_attention_f32(img, tok, d_lens, d_index, True)
    for _ in range(3):
        for o in out:
            o.fill_(7) if o.dtype == torch.int32 else o.fill_(-1.0)
        graph.replay()
        torch.cuda.synchronize()
        for o, e in zip(out, eager):
            assert o.shape == e.shape and torch.equal(o.view(torch.int32), e.view(torch.int32))
