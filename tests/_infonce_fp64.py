"""fp64 chain reference of the symmetric InfoNCE backward outside the one-kernel step: the multi-kernel flat step
(cvcl_flat_contrastive_step), the feature-level op (ops.sim_infonce_fwd / _bwd, one device or one shard) and the
sharded fallback of ops.flat_step_sharded.  All of them emit Gs = bf16(w (P_row + P_col)) with the diagonal included
(EpiGradG) and a per-row fp32 term gdiag = G_ii - bf16(Gs_ii), which the feature-gradient kernels add times the
positive.  Given the kernel's own bf16 features, LSEs, Gs and gdiag, infonce_chain returns what each of those
stages must produce, so a gate can name the stage that is off.

    infonce_chain(I, T, s, ...)   -- pure torch, any device (float64)
    normalize_bwd(q, g, inv)      -- the F.normalize backward
    diag_placements(I, T, s)      -- dI after the normalise backward with the diagonal of G in bf16 or in fp32

Test infrastructure (input builders and metrics: tests/_fused_fp64.py)."""
import math

import torch

D = torch.float64
# end-to-end worst row of a confident batch against fp64 (gradients after the normalise backward).  The diagonal of
# G in bf16 leaves ~0.15 (tests/test_infonce_fp64_host.py), in fp32 ~0.035: the gate keeps the two apart.
E2E_WORST_ROW = 6.5e-2


def normalize_bwd(q, g, inv):
    """d/dx of F.normalize(x) applied to g, with q = x/|x| and inv = 1/|x|"""
    return (g - q * (q * g).sum(1, keepdim=True)) * inv[:, None]


def infonce_chain(I, T, s, lse=None, Gs=None, gdiag=None, rows_bf16=True):
    """fp64 of every stage of the backward of the symmetric InfoNCE of logits exp(s) I T^T (one device, B pairs).

    I, T  [B,E]: the kernel's bf16 features (any dtype; promoted to float64)
    lse   (lse0 [B], lse1 [B]): the kernel's LSEs, which Gs and G_ii are formed from (None: the fp64 LSEs)
    Gs    the kernel's Gs0 [B,B] (dT then reads Gs0^T) or (Gs0, Gs1) with Gs1 the text-row orientation
          (None: bf16(w (P_row + P_col)) from `lse`)
    gdiag the kernel's per-row term, [B] or (gdiag0, gdiag1) (None: G_ii - Gs_ii of the Gs used)
    rows_bf16=False: no bf16 rounding of Gs (host tests): the chain is then the exact fp64 backward.
    Returns {name: float64 tensor}: S, lse0, lse1, loss, ent0, ent1, ds, ds_mag, Gs64 / Gs (from `lse`, before and
    after the bf16 rounding), Gii, gdiag
    (G_ii - Gs_ii per direction, [2,B]), dI, dT (before any normalise backward)."""
    I, T = I.to(D), T.to(D)
    B = I.shape[0]
    scale = math.exp(s)
    w = scale * 0.5 / B
    S = scale * (I @ T.t())
    r = dict(S=S)
    r["lse0"], r["lse1"] = torch.logsumexp(S, 1), torch.logsumexp(S, 0)
    dg = S.diagonal()
    P0, P1 = torch.softmax(S, 1), torch.softmax(S, 0)
    r["loss"] = 0.5 * ((r["lse0"] - dg).mean() + (r["lse1"] - dg).mean())
    r["ent0"] = (r["lse0"] - (P0 * S).sum(1)).mean()
    r["ent1"] = (r["lse1"] - (P1 * S).sum(0)).mean()
    eye = torch.eye(B, dtype=D, device=S.device)
    r["ds"] = ((w * (P0 + P1) - 2 * w * eye) * (S / scale)).sum()
    r["ds_mag"] = ((w * (P0 + P1) + 2 * w * eye) * (S / scale).abs()).sum()
    l0, l1 = (r["lse0"], r["lse1"]) if lse is None else (lse[0].to(D), lse[1].to(D))
    gs = w * (torch.exp(S - l0[:, None]) + torch.exp(S - l1[None, :]))
    r["Gs64"] = gs
    r["Gs"] = gs.to(torch.bfloat16).to(D) if rows_bf16 else gs
    # G_ii = w (P_row,ii - 1 + P_col,ii - 1): expm1, so that a confident pair keeps its relative accuracy
    r["Gii"] = w * (torch.expm1(dg - l0) + torch.expm1(dg - l1))
    if Gs is None:
        G0, G1 = r["Gs"], r["Gs"].t()
    elif isinstance(Gs, (tuple, list)):
        G0, G1 = Gs[0].to(D), Gs[1].to(D)
    else:
        G0 = Gs.to(D); G1 = G0.t()
    r["gdiag"] = torch.stack([r["Gii"] - G0.diagonal(), r["Gii"] - G1.diagonal()])
    if gdiag is None:
        gd0, gd1 = r["gdiag"][0], r["gdiag"][1]
    elif isinstance(gdiag, (tuple, list)):
        gd0, gd1 = gdiag[0].to(D), gdiag[1].to(D)
    else:
        gd0 = gd1 = gdiag.to(D)
    r["dI"] = G0 @ T + gd0[:, None] * T
    r["dT"] = G1 @ I + gd1[:, None] * I
    return r


def diag_placements(I, T, s):
    """image-side feature gradient after the normalise backward (unit rows, inv_norm 1), fp64 from the bf16
    features I, T: (exact, diagonal of G in bf16 with -2w added in fp32, diagonal of G in fp32)"""
    r = infonce_chain(I, T, s)
    I, T = I.to(D), T.to(D)
    w = math.exp(s) * 0.5 / I.shape[0]
    one = torch.ones(I.shape[0], dtype=D, device=I.device)
    exact = infonce_chain(I, T, s, rows_bf16=False)["dI"]
    bf16_diag = r["Gs"] @ T - 2 * w * T
    return tuple(normalize_bwd(I, g, one) for g in (exact, bf16_diag, r["dI"]))
