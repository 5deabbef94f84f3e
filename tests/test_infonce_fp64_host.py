"""CPU checks of the fp64 chain reference of the InfoNCE backward outside the one-kernel step (tests/_infonce_fp64.py):
without bf16 rounding it is the fp64 oracle step, and on confident pairs the committed end-to-end worst-row gate
tells the diagonal of G kept in fp32 from the diagonal rounded to bf16."""
import math

import pytest
import torch

import _fused_fp64 as F
import _infonce_fp64 as N
from _util import O, S_DEFAULT

D = torch.float64


def features(inp, normalize):
    """fp64 features of a flat step and their inverse norms"""
    x, W = torch.from_numpy(inp["f"]).to(D), torch.from_numpy(inp["W"]).to(D)
    u = x @ W.t() + torch.from_numpy(inp["b"]).to(D)
    inv_i = 1.0 / u.norm(dim=1) if normalize else torch.ones(u.shape[0], dtype=D)
    C = torch.from_numpy(F.counts(inp["ids"], inp["table"].shape[0]))
    lens = torch.from_numpy(inp["lens"]).to(D)
    txt, inv_t = F.text_features(C, torch.from_numpy(inp["table"]).to(D), lens, normalize)
    return x, u * inv_i[:, None], inv_i, txt, inv_t, C, lens


@pytest.mark.parametrize("B,normalize,s", [(8, True, S_DEFAULT), (13, True, 0.0), (9, False, 0.3), (1, True, S_DEFAULT),
                                           (1, False, math.log(100.0))])
def test_chain_without_rounding_equals_fp64_oracle(B, normalize, s):
    inp = F.random_inputs(40 + B, B, 16, 32, 40, L=7)
    if not normalize:
        inp["table"] *= 0.05
    x, img, inv_i, txt, inv_t, C, lens = features(inp, normalize)
    r = N.infonce_chain(img, txt, s, rows_bf16=False)
    du = N.normalize_bwd(img, r["dI"], inv_i) if normalize else r["dI"]
    dm = (N.normalize_bwd(txt, r["dT"], inv_t) if normalize else r["dT"]) / lens[:, None]
    ref = O.contrastive_step(torch.from_numpy(inp["f"]), torch.from_numpy(inp["ids"]), torch.from_numpy(inp["lens"]),
                             torch.from_numpy(inp["W"]), torch.from_numpy(inp["b"]), torch.from_numpy(inp["table"]),
                             s, "flat", normalize=normalize, dtype=D)
    assert abs(float(r["loss"] - ref["loss"])) <= 1e-10
    assert abs(float(r["ent0"] - ref["image_entropy"])) <= 1e-10
    assert abs(float(r["ent1"] - ref["text_entropy"])) <= 1e-10
    assert abs(float(r["ds"] - ref["ds"])) <= 1e-10 * (1 + abs(float(ref["ds"])))
    dtable = C.t() @ dm
    dtable[0] = 0
    for key, got in (("dW", du.t() @ x), ("db", du.sum(0)), ("dtable", dtable)):
        assert float((got - ref[key]).abs().max()) <= 1e-10 * (1 + float(ref[key].abs().max())), key
    if B == 1:
        # one pair: G = 0 exactly, and so is every gradient
        assert float(r["Gii"].abs().max()) <= 1e-15 and float(r["dI"].abs().max()) <= 1e-12


def test_chain_takes_the_kernels_blocks():
    """given Gs and gdiag, dI / dT are Gs T + gdiag o T and Gs1 I + gdiag1 o I, whatever the LSEs were"""
    g = torch.Generator().manual_seed(3)
    I = torch.nn.functional.normalize(torch.randn(6, 8, generator=g, dtype=D), dim=1)
    T = torch.nn.functional.normalize(torch.randn(6, 8, generator=g, dtype=D), dim=1)
    G0, G1 = torch.rand(6, 6, generator=g, dtype=D), torch.rand(6, 6, generator=g, dtype=D)
    g0, g1 = torch.randn(6, generator=g, dtype=D), torch.randn(6, generator=g, dtype=D)
    r = N.infonce_chain(I, T, 1.0, Gs=(G0, G1), gdiag=(g0, g1))
    assert torch.allclose(r["dI"], G0 @ T + g0[:, None] * T, rtol=0, atol=1e-14)
    assert torch.allclose(r["dT"], G1 @ I + g1[:, None] * I, rtol=0, atol=1e-14)
    r = N.infonce_chain(I, T, 1.0, Gs=G0)
    assert torch.allclose(r["gdiag"][1], r["Gii"] - G0.diagonal(), rtol=0, atol=0)


def test_worst_row_gate_needs_the_diagonal_in_fp32():
    """confident pairs (aligned_inputs: mean P_ii ~0.8) at B = E = 512, s = -log 0.07, on bf16 features: with the
    documented roundings (Gs in bf16), the diagonal of G kept in fp32 passes the committed worst-row gate (0.034)
    and the diagonal rounded to bf16 fails it (0.147)"""
    inp = F.aligned_inputs(512)
    _, img, _, txt, _, _, _ = features(inp, True)
    I, T = img.to(torch.bfloat16), txt.to(torch.bfloat16)
    exact, bf16_diag, fp32_diag = N.diag_placements(I, T, S_DEFAULT)
    assert F.worst_row(fp32_diag, exact) <= N.E2E_WORST_ROW
    assert F.worst_row(bf16_diag, exact) > 1.5 * N.E2E_WORST_ROW
