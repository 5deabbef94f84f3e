"""CPU: the reference forms the retrieval tests compare against, and the argument errors of the retrieval API (raised
before any device work)."""
import argparse

import numpy as np
import pytest
import torch

import multimodal_baby_b200 as cv
from _retrieval import scores_fp64, sorted_reference
from _util import O, S_DEFAULT, case_inputs, t


def _rows_with_ties_and_nans(rng, nq=40, nk=57):
    s = rng.standard_normal((nq, nk)).astype(np.float32)
    s[:, 5:9] = s[:, 1:2]                                            # exact ties
    s[::3, 20] = np.nan                                              # NaNs, two per row in some rows
    s[::5, 2] = np.nan
    s[1::4, 30] = 0.0
    s[1::4, 31] = -0.0                                               # -0 == +0
    s[2, :] = 1.0                                                    # a constant row
    s[3, :] = np.nan                                                 # an all-NaN row
    return s


@pytest.mark.parametrize("k", [1, 7, 57])
def test_sorted_reference_equals_stable_torch_sort(k):
    rng = np.random.RandomState(5)
    s = _rows_with_ties_and_nans(rng)
    order = torch.sort(torch.from_numpy(s), dim=1, descending=True, stable=True).indices.numpy()
    qg = rng.randint(0, 6, size=s.shape[0])
    kg = rng.randint(0, 6, size=s.shape[1])
    kg[kg == 5] = 4                                                  # group 5: queries without a positive
    topk, rank = sorted_reference(s, qg, kg, k)
    assert np.array_equal(topk, order[:, :k])
    for i in range(s.shape[0]):
        hits = np.flatnonzero(kg[order[i]] == qg[i])
        assert rank[i] == (hits[0] if hits.size else -1)
    assert (rank[qg == 5] == -1).all() and (rank[qg != 5] >= 0).all()
    # rank < k iff a positive is in the top-k
    assert np.array_equal(rank[rank >= 0] < k, (kg[topk] == qg[:, None]).any(axis=1)[rank >= 0])
    # pair mode: the positive of query i is key i
    topk, rank = sorted_reference(s, None, None, k)
    assert np.array_equal(rank, np.argmax(order == np.arange(s.shape[0])[:, None], axis=1))
    assert rank[3] == 3                                              # all-NaN row: index order


@pytest.mark.parametrize("sim", ["flat", "mean", "max"])
@pytest.mark.parametrize("normalize", [True, False])
def test_scores_fp64_agree_with_the_oracle_forward(sim, normalize):
    etype = "flat" if sim == "flat" else "spatial"
    inp = case_inputs(61, 6, 64, etype, Bt=9)
    f, ids, lens = t(inp["f"]), t(inp["ids"]), t(inp["lens"])
    lens[0] = 1; ids[0, 1:] = 0
    W, b, table = t(inp["W"]), t(inp["b"]), t(inp["table"])
    s64 = scores_fp64(sim, f, W, b, ids, lens, table, normalize)
    lpi, lpt, _, _ = O.forward(f, ids, lens, W, b, table, S_DEFAULT, etype, "mean" if sim == "flat" else sim, normalize)
    ref = lpi.double() / np.exp(S_DEFAULT)
    assert s64.shape == (6, 9)
    assert float((s64 - ref).abs().max()) <= 2e-6 * float(ref.abs().max())
    assert torch.equal(lpt, lpi.t())
    # head outputs instead of trunk features give the same scores
    u = O.head_flat(f.double(), W.double(), b.double()) if sim == "flat" else O.head_spatial(f.double(), W.double(),
                                                                                             b.double())
    assert torch.allclose(scores_fp64(sim, u, W, b, ids, lens, table, normalize, from_trunk_boundary=False), s64,
                          rtol=0, atol=1e-12)


def _lit(embedding_type, sim="max", E=64):
    args = argparse.Namespace(embedding_type=embedding_type, embedding_dim=E, normalize_features=True,
                              fix_temperature=True, temperature=0.07, text_encoder="embedding", sim=sim)
    vocab = {"<pad>": 0, "<unk>": 1, "<sos>": 2, "<eos>": 3, **{"w%d" % i: i for i in range(4, 50)}}
    return cv.MultiModalLitModel(cv.VisionEncoder(args, trunk="pooled"), cv.TextEncoder(vocab, 2048, args), args,
                                 vocab=vocab)


def test_evaluate_retrieval_rejects_bad_arguments_before_device_work():
    """CPU tensors: any device work would raise RuntimeError, so a ValueError shows the check comes first."""
    flat, spatial = _lit("flat"), _lit("spatial")
    ids, lens = torch.tensor([[2, 5, 3]] * 4), torch.tensor([3] * 4)
    f, maps = torch.zeros(4, 2048), torch.zeros(4, 2048, 7, 7)
    g4 = torch.arange(4)
    cases = [
        (flat, (torch.zeros(4, 2048, 7, 7), ids, lens), {}, r"\[N, 2048\]"),
        (flat, (torch.zeros(4, 64), ids, lens), {}, r"\[N, 2048\]"),
        (flat, (f, ids, lens), dict(from_trunk_boundary=False), r"\[N, 64\]"),
        (spatial, (f, ids, lens), {}, r"\[N, 2048, H, W\]"),
        (spatial, (torch.zeros(4, 2048, 7, 7), ids, lens), dict(from_trunk_boundary=False), r"\[N, 64, H, W\]"),
        (flat, (f, ids[0], lens), {}, "N_txt"),
        (flat, (f, ids, lens[:3]), {}, "N_txt"),
        (flat, (f[:3], ids, lens), {}, "pair mode"),
        (spatial, (maps[:3], ids, lens), {}, "pair mode"),
        (flat, (f, ids, lens), dict(frame_group=g4), "together"),
        (flat, (f, ids, lens), dict(text_group=g4), "together"),
        (flat, (f, ids, lens), dict(frame_group=g4[:3], text_group=g4), "frame_group"),
        (flat, (f, ids, lens), dict(frame_group=g4, text_group=g4.int()), "text_group"),
        (flat, (f, ids, lens), dict(k=0), "k=0"),
        (flat, (f, ids, lens), dict(k=5), r"\[1, 4\]"),
        (spatial, (maps, ids, lens), dict(k=2.0), "k=2.0"),
        (flat, (f, ids, lens), dict(recall_at=(1, 0)), "recall_at"),
        (flat, (f, ids, lens), dict(block_bytes=0), "block_bytes"),
    ]
    for lit, a, kw, match in cases:
        with pytest.raises(ValueError, match=match):
            lit.evaluate_retrieval(*a, **{"k": 2, **kw})
    # k is capped at 64 whatever the sizes
    big = torch.zeros(70, 2048)
    with pytest.raises(ValueError, match=r"\[1, 64\]"):
        flat.evaluate_retrieval(big, torch.tensor([[2, 5, 3]] * 70), torch.tensor([3] * 70), k=65)


def test_retrieval_op_rejects_bad_arguments_before_device_work():
    img, txt = torch.zeros(5, 49, 64), torch.zeros(5, 64)
    tok, lens = torch.zeros(5, 3, 64), torch.ones(5, dtype=torch.int64)
    with pytest.raises(ValueError, match="sim"):
        cv.ops.retrieval_f32(img, txt, None, "sum", True, 0.0)
    with pytest.raises(ValueError, match="flat features"):
        cv.ops.retrieval_f32(img, txt, None, "flat", True, 0.0)
    with pytest.raises(ValueError, match="pooled text factor"):
        cv.ops.retrieval_f32(img, tok, lens, "mean", True, 0.0)
    with pytest.raises(ValueError, match="per-token"):
        cv.ops.retrieval_f32(img, txt, lens, "max", True, 0.0)
    with pytest.raises(ValueError, match="lens"):
        cv.ops.retrieval_f32(img, tok, lens[:4], "max", True, 0.0)
    with pytest.raises(ValueError, match="pair mode"):
        cv.ops.retrieval_f32(img[:4], tok, lens, "max", True, 0.0)
    with pytest.raises(ValueError, match="k="):
        cv.ops.retrieval_f32(img, txt, None, "mean", True, 0.0, k=6)
    # valid arguments on CPU tensors reach the device check
    with pytest.raises(RuntimeError, match="CUDA"):
        cv.ops.retrieval_f32(img, txt, None, "mean", True, 0.0, k=5)
