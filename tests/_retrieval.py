"""Reference forms of the cross-modal retrieval evaluation (test infrastructure; may import oracle/).

`sorted_reference` states the order and rank rules literally: each query row sorted by (NaN first, value
descending, key index ascending), the torch.sort(descending=True, stable=True) order, and the rank of a query the
position of its first positive in that order.  `scores_fp64` restates the three score forms in fp64 from the oracle
heads and text encoders; `assert_within_near_ties` extends the near-tie rule of _spatial_eval to top-k lists and
rank counts."""
import numpy as np
import torch

from _spatial_eval import NEAR_TIE, match_fp64
from _util import O


def _np(x):
    return x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)


def retrieval_order(scores):
    """scores [Nq, Nk] -> int64 [Nq, Nk], the keys of every row in retrieval order."""
    s = _np(scores)
    idx = np.arange(s.shape[1])
    order = np.empty(s.shape, np.int64)
    for i, row in enumerate(s):
        nan = np.isnan(row)
        order[i] = np.lexsort((idx, -np.where(nan, 0, row), ~nan))     # last key first: NaN, -value, index
    return order


def sorted_reference(scores, q_group, k_group, k):
    """scores [Nq, Nk] full query rows (query i = row i); q_group [Nq] / k_group [Nk], or both None (pair mode: the
    positive of query i is key i).  -> (topk int64 [Nq, k], rank int64 [Nq], -1 for a query without a positive)."""
    order = retrieval_order(scores)
    nq = order.shape[0]
    if q_group is None:
        pos = order == np.arange(nq)[:, None]
    else:
        pos = _np(k_group)[order] == _np(q_group)[:, None]
    rank = np.where(pos.any(axis=1), pos.argmax(axis=1), -1)
    return order[:, :k], rank


def scores_fp64(sim, frames, W, b, ids, lens, table, normalize=True, from_trunk_boundary=True):
    """image->text scores [N_img, N_txt] in fp64 without the temperature (text->image is the transpose).
    frames: [N, 2048] trunk rows / [N, E] head outputs (flat), [N, 2048, H, W] layer4 maps / [N, E, H, W] head outputs
    (sim "mean" / "max")."""
    f = frames.double()
    if sim == "flat":
        u = O.head_flat(f, W.double(), b.double()) if from_trunk_boundary else f
        txt, _ = O.text_encoder_flat(ids, lens, table.double())
        if normalize:
            u, txt = O.l2_normalize(u, -1), O.l2_normalize(txt, -1)
        return u @ txt.t()
    u = O.head_spatial(f, W.double(), b.double()) if from_trunk_boundary else f
    return match_fp64(u, ids, lens, table, sim, normalize)


def assert_within_near_ties(topk, rank, s64, q_group, k_group, what=""):
    """topk / rank of an fp32 path against the fp64 scores s64 [Nq, Nk] of the same queries: the j-th key may differ
    from the fp64 order's j-th key only where their fp64 scores are within NEAR_TIE * max|row|, and a rank may differ
    from the fp64 rank by at most the number of keys within that band of the fp64 first positive's score.
    Returns the number of rows that differ."""
    s64 = _np(s64).astype(np.float64)
    topk, rank = _np(topk).astype(np.int64), _np(rank).astype(np.int64)
    ref_topk, ref_rank = sorted_reference(s64, q_group, k_group, topk.shape[1])
    differ = 0
    for i in range(s64.shape[0]):
        row = s64[i]
        tol = NEAR_TIE * np.abs(row).max()
        if not np.array_equal(topk[i], ref_topk[i]):
            differ += 1
            gap = np.abs(row[topk[i]] - row[ref_topk[i]]).max()
            assert gap < tol, "%s row %d: top-k %s vs fp64 %s, gap %.3e" % (what, i, topk[i], ref_topk[i], gap)
        if rank[i] != ref_rank[i]:
            differ += 1
            assert ref_rank[i] >= 0 and rank[i] >= 0, "%s row %d: rank %d vs fp64 %d" % (what, i, rank[i], ref_rank[i])
            p = retrieval_order(row[None])[0, ref_rank[i]]
            band = int((np.abs(row - row[p]) < tol).sum())
            assert abs(rank[i] - ref_rank[i]) < band, \
                "%s row %d: rank %d vs fp64 %d, %d keys in the near-tie band" % (what, i, rank[i], ref_rank[i], band)
    return differ
