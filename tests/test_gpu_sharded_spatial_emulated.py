"""-m gpu, ONE device: the sharded spatial "max" InfoNCE (ops.spatial_max_infonce) checked by running every rank's
share on the same GPU.  Rank r runs the arithmetic a real rank runs after its gathers (ops._spatial_max_block_fwd /
_spatial_max_block_bwd: spatial_max_fwd on the row block [b,N] and the column block [N,b], the block InfoNCE
entries with diag_off = r*b, spatial_max_bwd on both blocks) and is compared with the one-device path on the whole
batch.  The multi-GPU runs through a real process group are in tests/test_gpu_sharded_spatial.py."""
import math

import numpy as np
import pytest
import torch

from _sharded_spatial import ragged_batch
from _util import O, S_DEFAULT, assert_grad_close, rel_fro

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def cv():
    import multimodal_baby_b200 as m
    m._cabi.load()
    return m


def test_block_entries_equal_square_entries_at_world_1(cv):
    """b = N = B, diag_off = 0, both blocks the same matrix: bit-identical to cvcl_match_infonce_fwd / _bwd; the
    block backward's d scale is summed in a fixed order, so replays are bit-identical."""
    B = 1000
    gen = torch.Generator().manual_seed(3)
    match = (torch.randn(B, B, generator=gen) * 0.2 + 2.0 * torch.eye(B)).to(DEV)
    s = S_DEFAULT
    ops = cv.ops
    sq = ops._raw(ops.match_infonce_fwd)(match, s)
    bl = ops._raw(ops.match_infonce_block_fwd)(match, match, 0, s, 1.0 / B)
    assert torch.equal(sq[0][:5], bl[0][:5])                        # loss, accuracies, entropies
    for x, y in zip(sq[1:], bl[1:]):                                  # LSEs, arg-max
        assert torch.equal(x, y)
    _, lse0, lse1, _, _ = sq
    dm, ds_sq = ops._raw(ops.match_infonce_bwd)(match, s, lse0, lse1)
    dss = []
    for _ in range(3):
        dr, dc, ds = ops._raw(ops.match_infonce_block_bwd)(match, match, 0, s, 0.5 / B, lse0, lse1, lse0, lse1)
        assert torch.equal(dr, dm) and torch.equal(dc, dm)
        dss.append(ds.clone())
    assert all(torch.equal(d, dss[0]) for d in dss)
    assert abs(float(dss[0]) - float(ds_sq)) <= 1e-5 * abs(float(ds_sq)) + 1e-7
    with pytest.raises(ValueError):
        ops._raw(ops.match_infonce_block_fwd)(match[:10], match[:, :12], 0, s, 1.0 / B)


def _operands(cv, x, split):
    """what a rank gathers: the fp32 features (split) or their bf16 cast"""
    if split:
        return x.detach().float()
    n, k, E = x.shape
    return cv.ops.to_bf16_pair(x.reshape(n * k, E), False)[0].view(n, k, E)


def _emulated(cv, img, tok, lens, ids, Ls, world, s, split):
    """every rank's forward then backward (the LSE gathers done by hand) -> per-rank results"""
    ops = cv.ops
    B = img.shape[0]
    b = B // world
    Lm = tok.shape[1]
    gi, gt = _operands(cv, img, split), _operands(cv, tok, split)
    fwd = ops._spatial_max_block_fwd(split)
    ranks = []
    for r in range(world):
        sl = slice(r * b, (r + 1) * b)
        # the rank's own L, padded back to the longest L of all ranks as sharding.spatial_max_infonce_forward does
        tok_r = torch.cat([gt[sl, :Ls[r]], gt.new_zeros((b, Lm - Ls[r], gt.shape[2]))], 1)
        ids_r = torch.cat([ids[sl, :Ls[r]], ids.new_zeros((b, Lm - Ls[r]))], 1)
        out5, l0, l1, a0, a1, state = fwd(gi[sl], tok_r, lens[sl], ids_r, gi, gt, lens, ids, s, r * b, 1.0 / B)
        ranks.append(dict(out5=out5, lse0=l0, lse1=l1, a0=a0, a1=a1, state=state))
    lse0_all = torch.cat([q["lse0"] for q in ranks]); lse1_all = torch.cat([q["lse1"] for q in ranks])
    for r, q in enumerate(ranks):
        di, dt, ds = ops._spatial_max_block_bwd(q["state"], r * b, 0.5 / B, q["lse0"], lse1_all, lse0_all, q["lse1"])
        q.update(dimg=di, dtok=dt[:, :Ls[r]], ds=ds)
    return ranks


@pytest.mark.parametrize("split", [True, False], ids=["split_bf16", "bf16"])
@pytest.mark.parametrize("E", [64, 512])
@pytest.mark.parametrize("world,b", [(2, 20), (4, 10), (8, 128)])
def test_emulated_ranks_equal_single_gpu(cv, world, b, E, split):
    B = world * b
    img64, tok64, lens, ids, Ls = ragged_batch(11 + world, B, E, world)
    img = img64.float().to(DEV); tok = tok64.float().to(DEV); lens = lens.to(DEV); ids = ids.to(DEV)
    s = S_DEFAULT
    ops = cv.ops
    # one device, whole batch
    iv = img.clone().requires_grad_(True); tv = tok.clone().requires_grad_(True)
    sv = torch.tensor(s, device=DEV, requires_grad=True)
    match = ops.spatial_max_similarity(iv, tv, lens, ids, split=split)
    ref = ops.infonce_from_match(match, sv)
    ref[0].backward()
    _, lse0, lse1, _, _ = ops._raw(ops.match_infonce_fwd)(match.detach(), s)
    ranks = _emulated(cv, img, tok, lens, ids, Ls, world, s, split)
    for r, q in enumerate(ranks):
        sl = slice(r * b, (r + 1) * b)
        # the blocks are slices of the one-device match and the LSEs are the same numbers: exact
        assert torch.equal(q["state"][0], match.detach()[sl]), r
        assert torch.equal(q["state"][1], match.detach()[:, sl]), r
        assert torch.equal(q["lse0"], lse0[sl]) and torch.equal(q["lse1"], lse1[sl]), r
    tot = torch.stack([q["out5"] for q in ranks]).sum(0)
    for k in range(5):
        a, c = float(tot[k]), ref[k].item()
        assert abs(a - c) <= 2e-6 * max(1.0, abs(c)), (k, a, c)
    dimg = torch.cat([q["dimg"] for q in ranks])
    valid = torch.arange(tok.shape[1], device=DEV)[None, :] < lens[:, None]
    assert rel_fro(dimg.cpu().numpy(), iv.grad.cpu().numpy()) <= 1e-5
    for r, q in enumerate(ranks):
        sl = slice(r * b, (r + 1) * b)
        assert not q["dtok"][~valid[sl, :Ls[r]]].any()
    dtok = torch.cat([q["dtok"][valid[r * b:(r + 1) * b, :Ls[r]]] for r, q in enumerate(ranks)])
    assert rel_fro(dtok.cpu().numpy(), tv.grad[valid].cpu().numpy()) <= 1e-5
    ds = sum(float(q["ds"][0]) for q in ranks)
    assert abs(ds - sv.grad.item()) <= 1e-5 * abs(sv.grad.item()) + 1e-7
    if split:
        # against the oracle on the fp32 features (fp64 autograd of multimodal.py:771-822)
        i64 = img.double().requires_grad_(True); t64 = tok.double().requires_grad_(True)
        s64 = torch.tensor(s, dtype=torch.float64, device=DEV, requires_grad=True)
        m64 = O.similarity_spatial_max(i64.permute(0, 2, 1).reshape(B, E, 7, 7), t64, lens)
        lpi, lpt = O.logits_from_match(m64, s64)
        res = O.infonce(lpi.cpu(), lpt.cpu())                           # the oracle's labels live on the host
        res.loss.backward()
        assert abs(float(tot[0]) - res.loss.item()) <= 1e-3 * res.loss.item()
        assert_grad_close(dimg.cpu().numpy(), i64.grad.cpu().numpy(), "dimg")
        assert_grad_close(dtok.cpu().numpy(), t64.grad[valid].cpu().numpy(), "dtok")
        assert abs(ds - s64.grad.item()) <= 2e-2 * abs(s64.grad.item()) + 2e-3


def test_world8_b1024_beyond_one_gpu_backward(cv):
    """B = 8192 (world 8, b = 1024, L = 25, 7x7, E = 512): the one-device backward would need a 164 GB arg-max matrix.
    Forward of all 8 ranks, backward of two; LSEs of sampled rows / columns against fp64 on the bf16 features, the
    loss against its own LSE identity."""
    world, b, L, HW, E = 8, 1024, 25, 49, 512
    B = world * b
    gen = torch.Generator(device=DEV).manual_seed(8)
    img = torch.nn.functional.normalize(torch.randn(B, HW, E, device=DEV, generator=gen), dim=-1).to(torch.bfloat16)
    tok = torch.nn.functional.normalize(torch.randn(B, L, E, device=DEV, generator=gen), dim=-1)
    tok = (tok + 0.5 * img[:, :1].float()).to(torch.bfloat16)                     # correlated pairs
    rng = np.random.RandomState(8)
    ids_np, lens_np = O.synth_tokens(rng, B, L, 2350)
    lens = torch.from_numpy(lens_np).to(DEV); ids = torch.from_numpy(ids_np).to(DEV)
    valid = torch.arange(L, device=DEV)[None, :] < lens[:, None]
    tok = tok * valid[..., None]
    s = S_DEFAULT
    ops = cv.ops
    fwd = ops._spatial_max_block_fwd(False)
    outs, lse0, lse1, diag, keep = [], [], [], [], {}
    for r in range(world):
        sl = slice(r * b, (r + 1) * b)
        out5, l0, l1, _, _, state = fwd(img[sl], tok[sl], lens[sl], ids[sl], img, tok, lens, ids, s, r * b, 1.0 / B)
        outs.append(out5); lse0.append(l0); lse1.append(l1)
        diag.append(state[0][:, r * b:(r + 1) * b].diagonal().double())
        if r in (0, world - 1):
            keep[r] = state
        del state
    lse0 = torch.cat(lse0); lse1 = torch.cat(lse1); diag = torch.cat(diag)
    loss = float(torch.stack(outs).sum(0)[0])
    sc = math.exp(s)
    ident = float(0.5 * ((lse0.double() - sc * diag).mean() + (lse1.double() - sc * diag).mean()))
    assert abs(loss - ident) <= 1e-4 * abs(ident), (loss, ident)
    sel = torch.from_numpy(np.random.RandomState(9).choice(B, 64, replace=False)).to(DEV)
    tokd, imgd = tok.double(), img.double()
    rows = torch.cat([O.similarity_spatial_max(imgd[sel[k:k + 8]].permute(0, 2, 1).reshape(8, E, 7, 7), tokd, lens)
                      for k in range(0, 64, 8)])                                  # [64, B]
    cols = torch.cat([O.similarity_spatial_max(imgd[c:c + 1024].permute(0, 2, 1).reshape(-1, E, 7, 7), tokd[sel], lens[sel])
                      for c in range(0, B, 1024)])                                # [B, 64]
    assert float((lse0[sel].double() - torch.logsumexp(sc * rows, 1)).abs().max()) <= 2e-3
    assert float((lse1[sel].double() - torch.logsumexp(sc * cols, 0)).abs().max()) <= 2e-3
    del rows, cols, tokd, imgd
    for r, state in keep.items():
        torch.cuda.synchronize(); torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        di, dt, ds = ops._spatial_max_block_bwd(state, r * b, 0.5 / B, lse0[r * b:(r + 1) * b], lse1, lse0,
                                                 lse1[r * b:(r + 1) * b])
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        print("rank %d backward at B=%d: peak %.1f GB above the %.1f GB held before it" % (r, B, peak / 1e9, base / 1e9))
        assert di.shape == (b, HW, E) and dt.shape == (b, L, E)
        assert bool(torch.isfinite(di).all()) and bool(torch.isfinite(dt).all()) and math.isfinite(float(ds[0]))
        assert not dt[~valid[r * b:(r + 1) * b]].any()
