"""-m gpu: batched Labeled-S evaluation and category classification for spatial-embedding models (fp32 1x1-conv
head, spatial "max" scores, the factorised "mean" scores) against fp64 restatements and the reference's per-trial
loop.  Predictions follow the near-tie rule of tests/_spatial_eval.py; exact ties go to the lowest index."""
import argparse

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from _spatial_eval import assert_pred_within_near_ties, match_fp64, spatial_trial_loop
from _util import O, S_DEFAULT, case_inputs, t

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def cv():
    import multimodal_baby_b200 as m
    m._cabi.load()
    return m


def _spatial_lit(cv, sim, inp, E=512, normalize=True):
    args = argparse.Namespace(embedding_type="spatial", embedding_dim=E, normalize_features=normalize,
                              fix_temperature=True, temperature=0.07, text_encoder="embedding", sim=sim)
    vocab = {"<pad>": 0, "<unk>": 1, "<sos>": 2, "<eos>": 3, **{"w%d" % i: i for i in range(4, 2350)}}
    lit = cv.MultiModalLitModel(cv.VisionEncoder(args, trunk="pooled"), cv.TextEncoder(vocab, 2048, args), args,
                                vocab=vocab)
    with torch.no_grad():
        conv = lit.model.image_embed.model[-1]
        conv.weight.copy_(t(inp["W"])[:, :, None, None]); conv.bias.copy_(t(inp["b"]))
        lit.model.text_embed.embedding.weight.copy_(t(inp["table"]))
    return lit.to(DEV).eval()


@pytest.fixture(scope="module")
def trials():
    """256 seeded 4-way trials of 7x7 layer4 maps; two labels (lengths 3 and 1) shared through a
    staging.batch_trials-shaped label_index."""
    N = 256
    inp = case_inputs(4242, 8, 512, "spatial")
    rng = np.random.RandomState(4243)
    f = O.synth_trunk_features(rng, (N, 4, 2048, 7, 7))
    ids = np.zeros((2, 3), np.int64)
    ids[0] = [2, 1234, 3]
    ids[1, 0] = 777
    lens = np.array([3, 1], np.int64)
    index = rng.randint(0, 2, size=N).astype(np.int32)
    return dict(inp=inp, f=t(f), ids=t(ids), lens=t(lens), index=t(index))


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("B,HW,E", [(3, 49, 512), (5, 64, 64), (70, 1, 512), (2, 49, 64)])
def test_conv1x1_f32_matches_fp64(cv, B, HW, E):
    rng = np.random.RandomState(B * 1000 + HW + E)
    K = 2048
    H, W = (7, 7) if HW == 49 else ((8, 8) if HW == 64 else (1, 1))
    x = torch.from_numpy(np.maximum(rng.standard_normal((B, K, H, W)), 0).astype(np.float32))
    w = torch.from_numpy((rng.standard_normal((E, K)) / 45).astype(np.float32))
    b = torch.from_numpy(rng.standard_normal(E).astype(np.float32))
    got = cv.ops.conv1x1_f32(x.to(DEV), w.to(DEV), b.to(DEV))
    ref = F.conv2d(x.double(), w.double()[:, :, None, None], b.double()).permute(0, 2, 3, 1).reshape(B * HW, E)
    assert got.shape == (B * HW, E)
    assert float((got.cpu().double() - ref).abs().max()) <= 2e-5 * max(1.0, float(ref.abs().max()))
    # the [E,K,1,1] conv weight is accepted as is
    got4 = cv.ops.conv1x1_f32(x.to(DEV), w.to(DEV)[:, :, None, None], b.to(DEV))
    assert torch.equal(got, got4)


def _kernel_case(seed, M, E=512, HW=49, C=22, L=25):
    """image location rows and label token rows as the model hands them over: label lengths 1, 3 and 25 (and
    random ones in between), <pad> columns past the length."""
    rng = np.random.RandomState(seed)
    u = torch.from_numpy(rng.standard_normal((M, E, 7, 7)).astype(np.float32))
    table = torch.from_numpy(rng.standard_normal((2350, E)).astype(np.float32))
    table[0] = 0
    ids, lens = O.synth_tokens(rng, C, L, 2350, min_len=3)
    lens[0], lens[1], lens[2] = 1, 3, 25
    for c in range(3):
        ids[c] = 0
        ids[c, :lens[c]] = rng.randint(4, 2350, size=lens[c])
    return u, table, torch.from_numpy(ids), torch.from_numpy(lens)


@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("n_way", [4, 2])
def test_spatial_max_scores_both_modes_vs_fp64(cv, normalize, n_way):
    M = 24 * n_way
    u, table, ids, lens = _kernel_case(7 + n_way + 10 * normalize, M)
    tok, _ = cv.ops.text_features_spatial(ids.to(DEV), lens.to(DEV), table.to(DEV), normalize)
    img = u.permute(0, 2, 3, 1).reshape(M, 49, -1).to(DEV)
    ref = match_fp64(u, ids, lens, table, "max", normalize) * np.exp(S_DEFAULT)           # [M, C] logits
    # category mode: every image against the 22 labels
    pred, logits = cv.ops.classify_ncat_spatial(img, tok, lens.to(DEV), "max", normalize, S_DEFAULT)
    assert logits.shape == (M, 22) and pred.dtype == torch.int32
    assert float((logits.cpu().double() - ref).abs().max()) <= 2e-6 * float(ref.abs().max())
    assert_pred_within_near_ties(pred, torch.argmax(ref, dim=1), ref, "category")
    # trial mode: trial n scored against label index[n] (every label used, the long one included)
    N = M // n_way
    index = torch.arange(N, dtype=torch.int32) % 22
    pred, logits = cv.ops.eval_nway_spatial(img, tok, lens.to(DEV), index.to(DEV), n_way, "max", normalize, S_DEFAULT)
    ref_t = ref[torch.arange(M), index.long().repeat_interleave(n_way)].view(N, n_way)
    assert float((logits.cpu().double() - ref_t).abs().max()) <= 2e-6 * float(ref.abs().max())
    assert_pred_within_near_ties(pred, torch.argmax(ref_t, dim=1), ref_t, "trial")
    # predictions only: the same arg-max; a replay is bit-identical
    pred2, empty = cv.ops.eval_nway_spatial(img, tok, lens.to(DEV), index.to(DEV), n_way, "max", normalize,
                                            S_DEFAULT, False)
    assert empty.numel() == 0 and torch.equal(pred, pred2)
    _, logits2 = cv.ops.eval_nway_spatial(img, tok, lens.to(DEV), index.to(DEV), n_way, "max", normalize, S_DEFAULT)
    assert torch.equal(logits, logits2)


def test_mean_scores_past_65535_maps(cv):
    """the "mean" image factor pools more maps than one launch's grid holds (25 000 4-way trials = 100 000 maps)"""
    rng = np.random.RandomState(3)
    img = torch.from_numpy(rng.standard_normal((70000, 2, 8)).astype(np.float32)).to(DEV)
    txt = torch.from_numpy(rng.standard_normal((3, 8)).astype(np.float32)).to(DEV)
    pred, logits = cv.ops.classify_ncat_spatial(img, txt, torch.ones(3, dtype=torch.int64, device=DEV), "mean",
                                                False, 0.0)
    ref = img.double().sum(1) @ txt.double().t()
    assert float((logits.double() - ref).abs().max()) <= 2e-6 * float(ref.abs().max())
    assert_pred_within_near_ties(pred, torch.argmax(ref, dim=1), ref, "mean 70000")


# ------------------------------------------------------------------------------------------------ Lightning API
@pytest.mark.parametrize("sim", ["max", "mean"])
def test_evaluate_trials_spatial_vs_per_trial_loop(cv, trials, sim):
    inp = trials["inp"]
    lit = _spatial_lit(cv, sim, inp)
    f, ids, lens, index = trials["f"], trials["ids"], trials["lens"], trials["index"]
    pred, logits = lit.evaluate_trials(f.to(DEV), ids.to(DEV), lens.to(DEV), index.to(DEV))
    assert pred.shape == (256,) and logits.shape == (256, 4)
    rows = index.long()
    ref_pred, ref_logits = spatial_trial_loop(f, ids[rows], lens[rows], t(inp["W"]), t(inp["b"]), t(inp["table"]),
                                              S_DEFAULT, sim)
    np.testing.assert_allclose(logits.cpu().numpy(), ref_logits.numpy(), atol=5e-5)
    u = O.head_spatial(f.to(DEV).reshape(-1, 2048, 7, 7).double(), t(inp["W"], DEV).double(), t(inp["b"], DEV).double())
    s64 = match_fp64(u, ids.to(DEV), lens.to(DEV), t(inp["table"], DEV), sim)
    s64 = s64[torch.arange(1024, device=DEV), rows.to(DEV).repeat_interleave(4)].view(256, 4)
    assert_pred_within_near_ties(pred, ref_pred, s64, sim)
    assert 0 < int((pred == 0).sum()) < 256                          # random heads: a mixed set of answers
    # the same trials handed over as head outputs [N, 4, E, 7, 7] give the same answers
    w, b = lit.model._head()
    heads = cv.ops.conv1x1_f32(f.to(DEV).reshape(-1, 2048, 7, 7), w, b).view(256, 4, 7, 7, 512).permute(0, 1, 4, 2, 3)
    pred_h, logits_h = lit.evaluate_trials(heads, ids.to(DEV), lens.to(DEV), index.to(DEV), from_trunk_boundary=False)
    assert torch.equal(pred_h, pred) and torch.equal(logits_h, logits)


@pytest.mark.parametrize("sim", ["max", "mean"])
def test_evaluate_trials_spatial_exact_ties(cv, trials, sim):
    inp = trials["inp"]
    lit = _spatial_lit(cv, sim, inp)
    f = trials["f"][:64].clone()
    f[:, 2] = f[:, 0]                                                # the target duplicated at candidate 2
    ids, lens, index = trials["ids"].to(DEV), trials["lens"].to(DEV), trials["index"][:64].to(DEV)
    pred, logits = lit.evaluate_trials(f.to(DEV), ids, lens, index)
    assert torch.equal(logits[:, 0], logits[:, 2]) and not bool((pred == 2).any())
    best = logits.max(dim=1).values
    assert torch.equal(pred == 0, logits[:, 0] == best)
    # an all-zero map with a zero bias and normalisation on: every score is 0, the first candidate wins
    with torch.no_grad():
        lit.model.image_embed.model[-1].bias.zero_()
    pred, logits = lit.evaluate_trials(torch.zeros((3, 4, 2048, 7, 7), device=DEV), ids, lens, index[:3])
    assert float(logits.abs().max()) == 0.0 and pred.tolist() == [0, 0, 0]


@pytest.mark.parametrize("sim", ["max", "mean"])
def test_classify_frames_spatial_vs_reference_forward(cv, sim):
    inp = case_inputs(4300, 40, 512, "spatial")
    lit = _spatial_lit(cv, sim, inp)
    f = t(inp["f"])                                                  # [40, 2048, 7, 7]
    ids, lens = t(inp["ids"][:22]), t(inp["lens"][:22])
    pred, logits = lit.classify_frames(f.to(DEV), ids.to(DEV), lens.to(DEV))
    lpi, _, _, _ = O.forward(f, ids, lens, t(inp["W"]), t(inp["b"]), t(inp["table"]), S_DEFAULT, "spatial", sim)
    assert logits.shape == (40, 22) and pred.shape == (40,)
    np.testing.assert_allclose(logits.cpu().numpy(), lpi.numpy(), atol=5e-5)
    u = O.head_spatial(f.to(DEV).double(), t(inp["W"], DEV).double(), t(inp["b"], DEV).double())
    s64 = match_fp64(u, ids.to(DEV), lens.to(DEV), t(inp["table"], DEV), sim)
    assert_pred_within_near_ties(pred, torch.argmax(lpi, dim=1), s64, sim)


def test_validation_step_and_evaluate_trials_agree(cv, trials):
    """the Lightning per-trial step (split-bf16 head and scores) and the batched fp32 path answer the same 64
    spatial-max trials the same way, up to near-ties of the fp64 scores."""
    inp = trials["inp"]
    lit = _spatial_lit(cv, "max", inp)
    f, ids, lens, index = trials["f"][:64], trials["ids"], trials["lens"], trials["index"][:64]
    lit.log = lambda *a, **k: None
    acc = []
    with torch.no_grad():
        for n in range(64):
            r = int(index[n])
            batch = (f[n:n + 1].to(DEV), ids[r:r + 1].to(DEV), lens[r:r + 1].to(DEV), [["label%d" % r]])
            acc.append(lit.validation_step(batch, n, 1)["accuracy"])
    pred, _ = lit.evaluate_trials(f.to(DEV), ids.to(DEV), lens.to(DEV), index.to(DEV), want_logits=False)
    u = O.head_spatial(f.to(DEV).reshape(-1, 2048, 7, 7).double(), t(inp["W"], DEV).double(), t(inp["b"], DEV).double())
    s64 = match_fp64(u, ids.to(DEV), lens.to(DEV), t(inp["table"], DEV), "max")
    s64 = s64[torch.arange(256, device=DEV), index.long().to(DEV).repeat_interleave(4)].view(64, 4).cpu()
    for n in range(64):
        if acc[n] != int(pred[n] == 0):
            other = int(pred[n]) if acc[n] else 1 + int(torch.argmax(s64[n, 1:]))
            assert abs(float(s64[n, 0] - s64[n, other])) < 1e-6 * float(s64[n].abs().max()), n
