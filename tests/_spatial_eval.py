"""Reference forms of the spatial-embedding evaluation (test infrastructure; may import oracle/).

`spatial_trial_loop` is the reference's per-trial loop (eval.py:196-214, multimodal_lit.py:466-511) for a
spatial model: one oracle forward per trial on its n_way layer4 maps and its label.  `match_fp64` is a batched
fp64 restatement of the same scores (multimodal.py:757-780), used for the near-tie rule: a prediction may differ
from the reference's only where the reference's two candidates are within an fp32 near-tie, i.e. their fp64
scores differ by less than NEAR_TIE * max|score|."""
import torch
import torch.nn.functional as F

from _util import O

NEAR_TIE = 1e-6


def spatial_trial_loop(f_trials, ids, lens, W, b, table, s, sim, normalize=True):
    """f_trials [N, n_way, K, H, W]; ids / lens: the label row of every trial [N, L] / [N].
    -> (pred [N], logits_per_text[0] of every trial [N, n_way])."""
    preds, logits = [], []
    for n in range(f_trials.shape[0]):
        _, lpt, _, _ = O.forward(f_trials[n], ids[n:n + 1], lens[n:n + 1], W, b, table, s, "spatial", sim, normalize)
        preds.append(int(torch.argmax(lpt[0])))
        logits.append(lpt[0])
    return torch.tensor(preds), torch.stack(logits)


def match_fp64(u, ids, lens, table, sim, normalize=True):
    """u [M, E, H, W] head outputs, ids / lens [C, L] / [C] label rows -> match [M, C] in fp64 (no temperature)."""
    u = u.double()
    tok = table.double()[ids]                                        # <pad> rows are the zero row 0
    if normalize:
        u = F.normalize(u, dim=1)
        tok = F.normalize(tok, dim=-1)
    lens = lens.double()
    if sim == "mean":
        return torch.einsum("mehw,cle->mc", u, tok) / (u.shape[-2] * u.shape[-1] * lens)
    return torch.einsum("mehw,cle->mclhw", u, tok).amax(dim=(3, 4)).sum(dim=2) / lens


def assert_pred_within_near_ties(pred, ref_pred, scores64, what=""):
    """pred == ref_pred except where the two candidates' fp64 scores are within NEAR_TIE * max|score| of the row."""
    pred = torch.as_tensor(pred).long().cpu()
    ref_pred = torch.as_tensor(ref_pred).long().cpu()
    scores64 = scores64.double().cpu()
    bad = torch.nonzero(pred != ref_pred).flatten()
    for i in bad.tolist():
        row = scores64[i]
        gap = abs(float(row[pred[i]] - row[ref_pred[i]]))
        assert gap < NEAR_TIE * float(row.abs().max()), \
            "%s row %d: pred %d vs reference %d, fp64 gap %.3e" % (what, i, int(pred[i]), int(ref_pred[i]), gap)
    return len(bad)
