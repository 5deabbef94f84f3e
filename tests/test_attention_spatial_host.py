"""CPU: the fp64 reference of the spatial attention maps reduces to the model's own spatial scores, and the attention
map API rejects what it cannot map before any device work."""
import argparse

import numpy as np
import pytest
import torch

import multimodal_baby_b200 as cv
from _spatial_attention import spatial_attention_maps
from _spatial_eval import match_fp64


def _labels(rng, C, L, E, V=300):
    table = torch.from_numpy(rng.standard_normal((V, E)))
    table[0] = 0                                                     # <pad>, as nn.Embedding(padding_idx=0) keeps it
    lens = rng.randint(1, L + 1, size=C)
    lens[0] = 1
    ids = np.zeros((C, L), np.int64)
    for c in range(C):
        ids[c, :lens[c]] = rng.randint(4, V, size=lens[c])
    return table, torch.from_numpy(ids), torch.from_numpy(lens.astype(np.int64))


@pytest.mark.parametrize("normalize", [True, False])
def test_reference_maps_reduce_to_the_spatial_scores(normalize):
    """sim="max": sum_l max_p T / len; sim="mean": mean_p U -- both equal match_fp64 of the paired label to 1e-12."""
    rng = np.random.RandomState(5 + normalize)
    M, C, L, E = 12, 5, 9, 32
    u = torch.from_numpy(rng.standard_normal((M, E, 7, 7)))
    table, ids, lens = _labels(rng, C, L, E)
    index = torch.from_numpy(rng.randint(0, C, size=M))
    T, U = spatial_attention_maps(u, ids[index], lens[index], table, normalize)
    assert T.shape == (M, L, 7, 7) and U.shape == (M, 7, 7)
    live = torch.arange(L)[None, :] < lens[index][:, None]
    assert bool((T[~live] == 0).all())
    rows = torch.arange(M)
    ref_max = match_fp64(u, ids, lens, table, "max", normalize)[rows, index]
    ref_mean = match_fp64(u, ids, lens, table, "mean", normalize)[rows, index]
    got_max = T.amax(dim=(2, 3)).sum(dim=1) / lens[index].double()
    got_mean = U.mean(dim=(1, 2))
    scale = float(ref_max.abs().max())
    assert float((got_max - ref_max).abs().max()) <= 1e-12 * scale
    assert float((got_mean - ref_mean).abs().max()) <= 1e-12 * max(scale, float(ref_mean.abs().max()))


def _lit(embedding_type, E=64):
    args = argparse.Namespace(embedding_type=embedding_type, embedding_dim=E, normalize_features=True,
                              fix_temperature=True, temperature=0.07, text_encoder="embedding", sim="max")
    vocab = {"<pad>": 0, "<unk>": 1, "<sos>": 2, "<eos>": 3, **{"w%d" % i: i for i in range(4, 50)}}
    return cv.MultiModalLitModel(cv.VisionEncoder(args, trunk="pooled"), cv.TextEncoder(vocab, 2048, args), args,
                                 vocab=vocab)


def test_attention_map_api_rejects_what_it_cannot_map():
    ids, lens = torch.tensor([[2, 5, 3]]), torch.tensor([3])
    with pytest.raises(NotImplementedError, match="gradCAM"):
        _lit("flat").attention_maps(torch.zeros(1, 2048), ids, lens)
    with pytest.raises(NotImplementedError, match="gradCAM"):
        _lit("flat").model.spatial_attention_maps(torch.zeros(1, 2048), ids, lens)
    with pytest.raises(ValueError, match="layer4 map"):
        _lit("spatial").attention_maps(torch.zeros(1, 2048), ids, lens)          # pooled features, not a map

    op = cv.ops.spatial_attention_f32
    img, tok, lens = torch.zeros(8, 49, 64), torch.zeros(8, 5, 64), torch.ones(8, dtype=torch.int64)
    with pytest.raises(ValueError, match=r"\[M, HW, E\]"):
        op(img[0], tok, lens, None, True)
    with pytest.raises(ValueError, match="per-token"):
        op(img, tok[:, 0], lens, None, True)
    with pytest.raises(ValueError, match="per-token"):
        op(img, torch.zeros(8, 5, 32), lens, None, True)
    with pytest.raises(ValueError, match="lens"):
        op(img, tok, lens[:3], None, True)
    with pytest.raises(ValueError, match="text_index"):
        op(img, tok, lens, torch.zeros(3, dtype=torch.int32), True)
    with pytest.raises(ValueError, match="as many labels"):
        op(img, tok[:3], lens[:3], None, True)
