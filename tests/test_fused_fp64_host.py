"""CPU checks of the fp64 chain reference of the one-kernel flat step (tests/_fused_fp64.py) and of its input
builders: without bf16 rounding, the chain fed its own exact values is the fp64 oracle step."""
import math

import numpy as np
import pytest
import torch

import _fused_fp64 as F
from _util import O, S_DEFAULT


def exact_chain(inp, s, normalize):
    """run chain_reference stage by stage, feeding each phase the exact fp64 output of the one before"""
    D = torch.float64
    d = {k: torch.from_numpy(np.asarray(inp[k])) for k in ("ids", "lens")}
    d.update(x16=torch.from_numpy(inp["f"]).to(D), w16=torch.from_numpy(inp["W"]).to(D),
             b=torch.from_numpy(inp["b"]).to(D), table=torch.from_numpy(inp["table"]).to(D),
             C=torch.from_numpy(F.counts(inp["ids"], inp["table"].shape[0])))
    B, E = d["x16"].shape[0], d["table"].shape[1]
    z = torch.zeros(B, E, dtype=D)
    snap = dict(hpart=(d["x16"] @ d["w16"].t())[None], img16=z, txt16=z, invn=torch.ones(2, B, dtype=D),
                lse=torch.zeros(2, B, dtype=D), diag=torch.zeros(2, B, dtype=D), gdiag=torch.zeros(2, B, dtype=D),
                dq=torch.zeros(2, B, E, dtype=D), du16=z, dm16=z)
    r = F.chain_reference(d, snap, s, normalize, rows_bf16=False)
    snap.update(img16=r["img"], txt16=r["txt"], invn=torch.stack([r["invn_i"], r["invn_t"]]))
    r = F.chain_reference(d, snap, s, normalize, rows_bf16=False)
    snap.update(lse=torch.stack([r["lse0"], r["lse1"]]), diag=torch.stack([r["diag"], r["diag"]]))
    r = F.chain_reference(d, snap, s, normalize, rows_bf16=False)
    snap.update(dq=torch.stack([r["dq0"], r["dq1"]]), gdiag=torch.stack([r["gdiag"], r["gdiag"]]))
    r = F.chain_reference(d, snap, s, normalize, rows_bf16=False)
    snap.update(du16=r["du"], dm16=r["dm"])
    return F.chain_reference(d, snap, s, normalize, rows_bf16=False)


@pytest.mark.parametrize("B,normalize,s", [(8, True, S_DEFAULT), (13, True, 0.0), (9, False, 0.3), (1, True, S_DEFAULT)])
def test_exact_chain_equals_fp64_oracle(B, normalize, s):
    inp = F.random_inputs(3 + B, B, 16, 32, 40, L=7)
    if not normalize:
        inp["table"] *= 0.05
    r = exact_chain(inp, s, normalize)
    ref = O.contrastive_step(torch.from_numpy(inp["f"]), torch.from_numpy(inp["ids"]), torch.from_numpy(inp["lens"]),
                             torch.from_numpy(inp["W"]), torch.from_numpy(inp["b"]), torch.from_numpy(inp["table"]),
                             s, "flat", normalize=normalize, dtype=torch.float64)
    assert abs(float(r["loss"] - ref["loss"])) <= 1e-10
    assert abs(float(r["ent0"] - ref["image_entropy"])) <= 1e-10
    assert abs(float(r["ent1"] - ref["text_entropy"])) <= 1e-10
    assert abs(float(r["ds"] - ref["ds"])) <= 1e-10 * (1 + abs(float(ref["ds"])))
    for key in ("dW", "db", "dtable"):
        assert float((r[key] - ref[key]).abs().max()) <= 1e-10 * (1 + float(ref[key].abs().max())), key
    assert float((r["img"] - ref["image_features"]).abs().max()) <= 1e-12
    assert float((r["txt"] - ref["text_features"]).abs().max()) <= 1e-12


def test_chain_diagonal_replaced_in_p4():
    """the dQ of P3 holds Gs_ii t_i (Gs_ii = 2w at one pair); P4 replaces it by G_ii t_i = w (P_row,ii - 1 +
    P_col,ii - 1) t_i, which is 0 at one pair"""
    inp = F.random_inputs(5, 1, 16, 32, 40, L=7)
    r = exact_chain(inp, S_DEFAULT, True)
    w = math.exp(S_DEFAULT) * 0.5
    assert abs(float(r["gdiag"][0]) - 2 * w) <= 1e-12 and float(r["dq0"].abs().max()) > 0
    assert float(r["du"].abs().max()) <= 1e-12 and float(r["dm"].abs().max()) <= 1e-12


def test_aligned_inputs_confident_spread_and_duplicates():
    B = 512
    inp = F.aligned_inputs(B)
    assert inp["table"].shape[0] >= B + 4 and not inp["table"][[0, F.SOS, F.EOS]].any()
    img = O.encode_image(torch.from_numpy(F.bf16_round(inp["f"])).double(),
                         torch.from_numpy(F.bf16_round(inp["W"])).double(), torch.from_numpy(inp["b"]).double())
    txt, _ = O.encode_text(torch.from_numpy(inp["ids"]), torch.from_numpy(inp["lens"]),
                           torch.from_numpy(inp["table"]).double())
    cos = (img * txt).sum(1).numpy()
    np.testing.assert_allclose(cos, inp["a"], atol=1e-6)
    P = torch.softmax(math.exp(S_DEFAULT) * img @ txt.t(), 1).diagonal().numpy()
    firm = P[:-6]                                   # before the loose pairs
    assert firm.min() < 0.35 and 0.3 <= np.quantile(firm, 0.02) and firm.max() > 0.99
    assert P[-6:].max() < 0.2                         # loose pairs: the arg-max lies among unrelated columns
    # exact duplicates, one per merge level of the arg-max
    lv = inp["dups"]
    assert set(lv) == {"chunk", "half", "tile", "block"}
    for i, j in lv.values():
        assert i < j and inp["f"][i].tobytes() == inp["f"][j].tobytes()
        assert inp["ids"][i].tobytes() == inp["ids"][j].tobytes() and inp["lens"][i] == inp["lens"][j]
    (a, b), (c, d), (e, f), (g, h) = lv["chunk"], lv["half"], lv["tile"], lv["block"]
    assert a // 32 == b // 32
    assert c // 64 == d // 64 and c // 32 != d // 32
    assert e // 128 == f // 128 and e // 64 != f // 64
    assert g // 128 != h // 128
    # every other pair has a token of its own
    own = inp["ids"][:, 1]
    assert len(set(own.tolist())) == B - len(lv)


def test_long_tiny_vocab_and_count_builders():
    long = F.long_inputs(64, 128, 64, 2350, L=77)
    assert long["ids"].shape == (64, 77) and long["lens"].max() > 64
    C, early = F.counts(long["ids"], 2350), F.counts(long["ids"][:, :32], 2350)
    assert ((C > early) & (early > 0)).sum(1).min() > 0          # every row repeats a token across chunks
    tiny = F.random_inputs(1, 640, 384, 1024, 6)
    Ct = F.counts(tiny["ids"], 6)
    assert (Ct.max(1) > 1).mean() > 0.8
    c = F.count257_inputs(128, 512, 64, 2350)
    Cc = F.counts(c["ids"], 2350)
    assert c["ids"].shape[1] == 260 and Cc[0, c["tok_v"]] == 257 and Cc[0, c["tok_u"]] == 1
    assert Cc[1:, c["tok_v"]].sum() == 0 and Cc[1:, c["tok_u"]].sum() == 0
    assert int(c["lens"][0]) == 260 and (c["ids"][1:, 25:] == 0).all()
