"""CPU: the reference forms the spatial evaluation tests compare against, and the shape errors of the spatial
evaluation API (raised before any device work)."""
import argparse

import numpy as np
import pytest
import torch

import multimodal_baby_b200 as cv
from _spatial_eval import NEAR_TIE, match_fp64, spatial_trial_loop
from _util import O, S_DEFAULT, case_inputs, t


@pytest.mark.parametrize("sim", ["max", "mean"])
@pytest.mark.parametrize("normalize", [True, False])
def test_spatial_trial_loop_equals_batched_fp64(sim, normalize):
    """the per-trial loop (one oracle forward per trial, fp32) == the batched fp64 scores, label rows with
    <pad> columns past their lengths."""
    inp = case_inputs(31, 6, 64, "spatial")
    rng = np.random.RandomState(32)
    N = 6
    f = t(O.synth_trunk_features(rng, (N, 4, 2048, 7, 7)))
    ids, lens = t(inp["ids"]), t(inp["lens"])                        # [6, 25]: lengths 3..25, pads after
    lens[0] = 1; ids[0, 1:] = 0
    pred, logits = spatial_trial_loop(f, ids, lens, t(inp["W"]), t(inp["b"]), t(inp["table"]), S_DEFAULT, sim,
                                      normalize)
    u = O.head_spatial(f.reshape(-1, 2048, 7, 7).double(), t(inp["W"]).double(), t(inp["b"]).double())
    s64 = match_fp64(u, ids, lens, t(inp["table"]), sim, normalize)    # [N*4, N]: every image against every label
    s64 = s64[torch.arange(4 * N), torch.arange(N).repeat_interleave(4)].view(N, 4) * np.exp(S_DEFAULT)
    assert logits.shape == (N, 4)
    assert float((logits.double() - s64).abs().max()) <= 2e-6 * float(s64.abs().max())
    for n in range(N):
        best = int(torch.argmax(s64[n]))
        assert int(pred[n]) == best or abs(float(s64[n, best] - s64[n, pred[n]])) < NEAR_TIE * float(s64[n].abs().max())


def _spatial_lit(sim="max", E=64):
    args = argparse.Namespace(embedding_type="spatial", embedding_dim=E, normalize_features=True, fix_temperature=True,
                              temperature=0.07, text_encoder="embedding", sim=sim)
    vocab = {"<pad>": 0, "<unk>": 1, "<sos>": 2, "<eos>": 3, **{"w%d" % i: i for i in range(4, 50)}}
    return cv.MultiModalLitModel(cv.VisionEncoder(args, trunk="pooled"), cv.TextEncoder(vocab, 2048, args), args,
                                 vocab=vocab)


def test_spatial_model_rejects_pooled_and_misshapen_features():
    lit = _spatial_lit()
    ids, lens = torch.tensor([[2, 5, 3]]), torch.tensor([3])
    with pytest.raises(ValueError, match=r"\[N, 4, 2048, H, W\]"):
        lit.evaluate_trials(torch.zeros(2, 4, 2048), ids, lens, torch.zeros(2, dtype=torch.int32))
    with pytest.raises(ValueError, match=r"\[N, 4, 64, H, W\]"):
        lit.evaluate_trials(torch.zeros(2, 4, 2048, 7, 7), ids, lens, from_trunk_boundary=False)
    with pytest.raises(ValueError, match=r"\[N, 4, 2048, H, W\]"):
        lit.evaluate_trials(torch.zeros(2, 3, 2048, 7, 7), ids, lens)           # 3 candidates, n_way = 4
    with pytest.raises(ValueError, match=r"\[N, 2048, H, W\]"):
        lit.classify_frames(torch.zeros(5, 2048), ids, lens)


def test_eval_ops_reject_shapes_that_do_not_fit():
    with pytest.raises(ValueError, match="do not fit"):
        cv.ops.linear_f32(torch.zeros(3, 2048), torch.zeros(8, 512), None)
    with pytest.raises(ValueError, match="bias"):
        cv.ops.linear_f32(torch.zeros(3, 16), torch.zeros(8, 16), torch.zeros(9))
    with pytest.raises(ValueError):
        cv.ops.conv1x1_f32(torch.zeros(1, 2048, 7, 7), torch.zeros(64, 1024), None)
    img, tok, lens = torch.zeros(8, 49, 64), torch.zeros(3, 5, 64), torch.ones(3, dtype=torch.int64)
    with pytest.raises(ValueError, match="per-token"):
        cv.ops.eval_nway_spatial(img, tok[:, 0], lens, None, 4, "max", True, 0.0)
    with pytest.raises(ValueError, match="pooled text factor"):
        cv.ops.eval_nway_spatial(img, tok, lens, None, 4, "mean", True, 0.0)
    with pytest.raises(ValueError, match="n_way"):
        cv.ops.eval_nway_spatial(img, tok, lens, None, 3, "max", True, 0.0)
    with pytest.raises(ValueError, match="txt_index"):
        cv.ops.eval_nway_spatial(img, tok, lens, torch.zeros(3, dtype=torch.int32), 4, "max", True, 0.0)
    with pytest.raises(ValueError, match="sim"):
        cv.ops.classify_ncat_spatial(img, tok, lens, "sum", True, 0.0)
