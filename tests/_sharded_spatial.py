"""fp64 torch restatement of one rank's arithmetic of the sharded spatial "max" InfoNCE (the `compute_fwd` /
`compute_bwd` that sharding.spatial_max_infonce_forward / _backward take; on the GPU ops.py passes the CUDA
kernels), plus the shared synthetic batch of the sharded spatial tests."""
import math

import torch


def spatial_max64(img, tok, lens):
    """match[i,t] = sum_{l < len[t]} max_hw <img[i,hw], tok[t,l]> / len[t]; img [Bi,HW,E], tok [Bt,L,E]."""
    sc = torch.einsum('ihe,tle->itlh', img.double(), tok.double()).amax(-1)          # [Bi, Bt, L]
    valid = torch.arange(tok.shape[1], device=lens.device)[None, :] < lens[:, None]   # [Bt, L]
    return (sc * valid[None]).sum(-1) / lens[None].double()


def _ce_stats(x, diag_off):
    """x [b, N] logits of b queries whose positive sits at column m + diag_off."""
    lse = torch.logsumexp(x, 1)
    idx = torch.arange(x.shape[0])
    ce = (lse - x[idx, idx + diag_off]).sum()
    ent = (lse - (torch.softmax(x, 1) * x).sum(1)).sum()
    arg = x.argmax(1)
    return lse, ce, ent, (arg == idx + diag_off).sum().double(), arg


def compute_fwd(img_r, tok_r, lens_r, ids_r, img_all, tok_all, lens_all, ids_all, ls, diag_off, inv_rows):
    assert tok_r.shape[1] == tok_all.shape[1]                      # padded to the longest L of all ranks
    if ids_all is not None:
        assert tuple(ids_all.shape) == tuple(tok_all.shape[:2])
    sc = math.exp(ls)
    match_r = spatial_max64(img_r, tok_all, lens_all)              # [b, N]
    match_c = spatial_max64(img_all, tok_r, lens_r)                # [N, b]
    lse0, ce0, ent0, acc0, a0 = _ce_stats(sc * match_r, diag_off)
    lse1, ce1, ent1, acc1, a1 = _ce_stats(sc * match_c.t(), diag_off)
    out5 = torch.zeros(8, dtype=torch.float64)
    out5[0] = (ce0 + ce1) * 0.5 * inv_rows
    out5[1] = acc0 * inv_rows; out5[2] = acc1 * inv_rows
    out5[3] = ent0 * inv_rows; out5[4] = ent1 * inv_rows
    state = (img_r, tok_r, lens_r, img_all, tok_all, lens_all, match_r, match_c, ls)
    return out5, lse0, lse1, a0.int(), a1.int(), state


def compute_bwd(state, diag_off, coef, lse0, lse1_all, lse0_all, lse1):
    img_r, tok_r, lens_r, img_all, tok_all, lens_all, match_r, match_c, ls = state
    sc = math.exp(ls)
    b = img_r.shape[0]
    idx = torch.arange(b)
    xr = sc * match_r
    g_r = coef * (torch.exp(xr - lse0[:, None]) + torch.exp(xr - lse1_all[None, :]))
    g_r[idx, idx + diag_off] -= 2 * coef
    xc = sc * match_c
    g_c = coef * (torch.exp(xc - lse0_all[:, None]) + torch.exp(xc - lse1[None, :]))
    g_c[idx + diag_off, idx] -= 2 * coef
    ir = img_r.double().clone().requires_grad_(True)
    (spatial_max64(ir, tok_all, lens_all) * (sc * g_r)).sum().backward()
    tr = tok_r.double().clone().requires_grad_(True)
    (spatial_max64(img_all, tr, lens_r) * (sc * g_c)).sum().backward()
    return ir.grad, tr.grad, (g_r * xr).sum().reshape(1)


def ragged_batch(seed, B, E, world, HW=49, V=2350):
    """(img [B,HW,E], tok [B,Lmax,E], lens [B], ids [B,Lmax], L per rank): unit-norm fp64 features, zero token rows
    and <pad> ids beyond len; rank r's rows have their longest utterance at L_r = 4 + 3r (all L_r differ)."""
    g = torch.Generator().manual_seed(seed)
    b = B // world
    Ls = [4 + 3 * r for r in range(world)]
    Lm = max(Ls)
    lens = torch.cat([torch.cat([torch.tensor([L]), torch.randint(1, L + 1, (b - 1,), generator=g)]) for L in Ls])
    img = torch.nn.functional.normalize(torch.randn(B, HW, E, generator=g, dtype=torch.float64), dim=-1)
    tok = torch.nn.functional.normalize(torch.randn(B, Lm, E, generator=g, dtype=torch.float64), dim=-1)
    img[:, :, 0] += 0.3 * tok[:, :1, 0]                                  # correlated pairs
    valid = torch.arange(Lm)[None, :] < lens[:, None]
    tok = tok * valid[..., None]
    ids = torch.randint(4, V, (B, Lm), generator=g) * valid
    return img, tok, lens, ids, Ls
