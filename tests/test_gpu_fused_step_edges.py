"""The one-kernel flat step (csrc/fused_step.cuh) at the branches of its plan that the default shape never takes,
and in the confident-softmax regime of a trained model, every phase against the fp64 chain reference of
tests/_fused_fp64.py (fp64 from the kernel's own output of the previous phase).

Each case first asserts, from ops.fused_layout, the plan property it exists to cover, so a later plan change
cannot move it off its branch silently.  Then, for every case: the phase gates, no NaN, five bit-identical
replays, the control block back at zero and, where the sharded plan admits the shape, the sharded instance at
world 1 bit-identical to the single-GPU one.

The committed gates are about 4x the worst errors measured on a B200; DESIGN section 4 lists both.
Set FUSED_EDGES_REPORT=<file> to append every case's measured values to <file> as JSON lines."""
import math

import numpy as np
import pytest
import torch

import _fused_fp64 as F
from _util import O, S_DEFAULT, cosine, rel_fro

pytestmark = pytest.mark.gpu
DEV = "cuda"

# gates (fp64 chain, see DESIGN section 4)
GATE = dict(                # measured maximum over the cases on a B200 (1000 W) in brackets
    head_row=2e-6,          # P0 slab sum + bias vs x16 w16^T + b, worst row            [4.4e-7]
    feat_abs=1e-6,          # img_f32 / txt_f32 max abs                                 [2.1e-7]
    invn_rel=1e-6,          #                                                           [1.6e-7]
    lse_abs=5e-5,           # both LSE arrays                                           [1.3e-5]
    diag_abs=4e-5,          #                                                           [8.7e-6]
    part_m_abs=6e-5,        # per-partial row maxima                                    [1.5e-5]
    loss_rel=8e-6,          #                                                           [2.0e-6]
    ent_abs=1.2e-5,         #                                                           [2.9e-6]
    dq_row=2e-3,            # dQ slab sums vs bf16(Gs) K, worst row                     [4.5e-4]
    ds_rel=2e-6,            # |ds - ref| / sum |G| |S|                                  [4.2e-7]
    p4_ulp=16.0,            # du16 / dm16 in bf16 ulps (floor: 2^-20 of the row max)    [4.0]
    db_rel=1.5e-6,          # |db - ref| / sum_r |du_r|                                 [3.6e-7]
    dw_row=7e-6,            #                                                           [1.7e-6]
    dt_row=3e-7,            #                                                           [6.7e-8]
)
NEAR_TIE = 1e-6             # DESIGN section 4: an fp64 top-two gap below 1e-6 max|S| may go either way


def Gates(name):
    return F.Gates(name, "FUSED_EDGES_REPORT")


@pytest.fixture(scope="module")
def cv():
    import multimodal_baby_b200 as m
    m._cabi.load()
    return m


@pytest.fixture(autouse=True)
def _natural_plan(monkeypatch):
    monkeypatch.delenv("CVCL_B200_FUSED_FORCE_T", raising=False)
    monkeypatch.delenv("CVCL_B200_FUSED_FORCE_QS", raising=False)


def natural_t2_batch(cv):
    """the largest batch the plan takes with two similarity tiles per CTA (1536 on 148 SMs)"""
    lib = cv._cabi.load()
    for nmb in range(32, 0, -1):
        B = 128 * nmb
        if lib.cvcl_flat_fused_supported(B, 25, 512, 2048, 2350):
            lay = cv.ops.fused_layout(B, 25, 512, 2048, 2350)
            assert lay["nCB"] // lay["nPart"] == 2, lay
            return B
    raise AssertionError("no batch with T = 2")


def check_chain(cv, g, inp, d, sn, s, normalize=True):
    """every phase gate of one captured step"""
    lay = sn["lay"]
    B, E = d["x16"].shape[0], d["table"].shape[1]
    r = F.chain_reference(d, sn, s, normalize)
    # ---- P0 / P1
    g.le("P0 head worst row", F.worst_row(sn["hpart"].double().sum(0) + d["b"].double(), r["u"]), GATE["head_row"])
    g.le("P0 txt_f32 max abs", (sn["txt_f"].double() - r["txt"]).abs().max(), GATE["feat_abs"])
    g.le("P1 img_f32 max abs", (sn["img_f"].double() - r["img"]).abs().max(), GATE["feat_abs"])
    g.true("P0 txt16 == bf16(txt_f32)", torch.equal(sn["txt16"], sn["txt_f"].bfloat16()))
    g.true("P1 img16 == bf16(img_f32)", torch.equal(sn["img16"], sn["img_f"].bfloat16()))
    g.le("P0 invn_t rel", ((sn["invn"][1].double() - r["invn_t"]) / r["invn_t"]).abs().max(), GATE["invn_rel"])
    g.le("P1 invn_i rel", ((sn["invn"][0].double() - r["invn_i"]) / r["invn_i"]).abs().max(), GATE["invn_rel"])
    g.true("P1 counts exact", torch.equal(sn["cmat"].double(), d["C"]))
    # ---- P2 / P3
    g.le("P3 lse0 max abs", (sn["lse"][0].double() - r["lse0"]).abs().max(), GATE["lse_abs"])
    g.le("P3 lse1 max abs", (sn["lse"][1].double() - r["lse1"]).abs().max(), GATE["lse_abs"])
    g.le("P2 diag max abs", (sn["diag"].double() - r["diag"][None]).abs().max(), GATE["diag_abs"])
    S = r["S"]
    tol = NEAR_TIE * float(S.abs().max())
    bad_arg = 0; m_err = 0.0
    for z, Sz in enumerate((S, S.t())):
        for pi in range(sn["part_m"].shape[1]):
            c0, c1 = 64 * pi, min(B, 64 * pi + 64)
            if c0 >= B:
                break
            arg, gap = F.first_argmax_and_gap(Sz[:, c0:c1])
            karg = sn["part_arg"][z, pi].long() - c0
            near = (gap > 0) & (gap < tol)
            bad_arg += int(((karg != arg) & ~near).sum())
            m_err = max(m_err, float((sn["part_m"][z, pi].double() - Sz[:, c0:c1].max(1).values).abs().max()))
    g.true("P2 partial arg-max (first index)", bad_arg == 0, bad_arg)
    g.le("P2 partial max abs", m_err, GATE["part_m_abs"])
    out5 = sn["out5"].double()
    if B > 1:                                   # (B = 1: the loss is 0, see test_fused_branch_vs_fp64_chain)
        g.le("loss rel", abs(out5[0] - r["loss"]) / abs(float(r["loss"])), GATE["loss_rel"])
    g.le("image entropy abs", abs(out5[3] - r["ent0"]), GATE["ent_abs"])
    g.le("text entropy abs", abs(out5[4] - r["ent1"]), GATE["ent_abs"])
    # exact duplicates decided across two partials: the first index must win if the kernel's two partial maxima are
    # bit-equal; if its S columns differ after all (MMA rounding by tile position), those rows follow the near-tie rule
    excuse = torch.zeros(2, B, dtype=torch.bool, device=S.device)
    for lvl, (i, j) in (inp.get("dups") or {}).items():
        if i // 64 == j // 64:
            continue
        for z in range(2):
            for row in (i, j):
                eq = bool(sn["part_m"][z, i // 64, row] == sn["part_m"][z, j // 64, row])
                g.values["dup %s z%d row %d: partial maxima bit-equal" % (lvl, z, row)] = eq
                if not eq:
                    excuse[z, row] = True
    acc = F.accuracy_bounds(S, lay["Bp"] // 128, NEAR_TIE, excuse)
    kacc = sn["rb_part"][:, :, 4:6].cpu().numpy()
    ok = True
    for z in range(2):
        for rb in range(acc.shape[1]):
            c = kacc[z, rb, z]
            ok = ok and acc[z, rb, 0] <= c <= acc[z, rb, 0] + acc[z, rb, 1]
    g.true("P3 accuracy per row block (exact up to near-ties)", ok,
           "kernel %s ref(sure, near) %s" % (kacc[..., 0].tolist() + kacc[..., 1].tolist(), acc.tolist()))
    # the recorded diagonal is the bf16 rounding of Gs_ii (one bf16 ulp of fp64 from the kernel's LSEs)
    gd = sn["gdiag"].double()
    g.true("P3 gdiag bf16-representable", torch.equal(sn["gdiag"], sn["gdiag"].bfloat16().float()))
    g.le("P3 gdiag ulps", ((gd - r["gdiag"][None]).abs() / F.bf16_ulp(r["gdiag"][None])).max(), 1.0)
    g.le("P3 dI worst row", F.worst_row(sn["dq"][0], r["dq0"]), GATE["dq_row"])
    g.le("P3 dT worst row", F.worst_row(sn["dq"][1], r["dq1"]), GATE["dq_row"])
    g.le("P3 ds rel", F.rel_to(float(sn["ds"][0]) - float(r["ds"]), r["ds_mag"]), GATE["ds_rel"])
    # ---- P4: within one bf16 ulp of fp64 from the kernel's own dQ sums
    for key, ref in (("du16", r["du"]), ("dm16", r["dm"])):
        floor = 2.0 ** -20 * ref.abs().amax(1, keepdim=True)
        ulps = (sn[key].double() - ref).abs() / torch.maximum(F.bf16_ulp(ref), floor)
        g.le("P4 %s max ulps" % key, ulps.max(), GATE["p4_ulp"])
    g.le("P4 db rel", F.rel_to((sn["db"].double() - r["db"]).abs().max(), r["db_mag"].max()), GATE["db_rel"])
    # ---- P5
    g.le("P5 dW worst row", F.worst_row(sn["dW"], r["dW"]), GATE["dw_row"])
    present = d["C"].sum(0) > 0
    g.le("P5 dtable worst row", F.worst_row(sn["dtable"][present], r["dtable"][present]), GATE["dt_row"])
    g.true("P5 dtable absent rows and row 0 exactly 0", not bool(sn["dtable"][~present].any()))
    # ---- every case
    g.true("no NaN", not bool(torch.isnan(sn["flat"][:1]).any() or torch.isnan(sn["flat"][4:]).any()
                              or torch.isnan(sn["out5"][:5]).any()))
    g.true("5 replays bit-identical", sn["replays_identical"])
    g.true("control block zero", sn["ctrl"][:3] == [0, 0, 0], sn["ctrl"][:3])
    return r


def check_sharded(cv, g, d, sn, s, normalize=True):
    B, K = d["x16"].shape
    if B % 128 or K % 128:
        return
    o, flat = F.sharded_world1(cv, d, s, normalize)
    g.true("sharded world 1 bit-identical", torch.equal(o[:5], sn["out5"][:5]) and torch.equal(flat[:1], sn["flat"][:1])
           and torch.equal(flat[4:], sn["flat"][4:]))


def run_case(cv, name, inp, s=S_DEFAULT, normalize=True, s_dev=False, prop=None):
    g = Gates(name)
    d = F.device_inputs(inp, DEV)
    B, K = d["x16"].shape; V, E = d["table"].shape; L = d["ids"].shape[1]
    pl = F.plan(cv.ops.fused_layout(B, L, E, K, V), B, E, K, V)
    if prop is not None:
        assert prop(pl), "%s: plan %s is not on the branch this case covers" % (name, pl)
    sd = torch.tensor(s, dtype=torch.float32, device=DEV) if s_dev else None
    sn = F.capture(cv, d, s, normalize, s_dev=sd)
    r = check_chain(cv, g, inp, d, sn, s, normalize)
    check_sharded(cv, g, d, sn, s, normalize)
    return g, d, sn, r


# name, B, L, E, K, V, plan property
SHAPES = [
    ("p5_multitile", 512, 25, 512, 2048, 8192, lambda p: p["p5_tiles"] > p["grid"] - 1),
    ("dw_bn64", 300, 25, 512, 576, 2350, lambda p: p["dw_bn"] == 64),
    ("kc1_ks1_bn64", 256, 25, 256, 64, 2350, lambda p: p["num_kc"] == 1 and p["KS"] == 1 and p["dw_bn"] == 64),
    ("neb1_qs1", 256, 25, 128, 2048, 2350, lambda p: p["nEB"] == 1 and p["QS"] == 1),
    ("ragged_b1", 1, 25, 512, 2048, 2350, lambda p: p["nMB"] == 1),
    ("ragged_b2", 2, 25, 512, 2048, 2350, lambda p: p["nMB"] == 1),
    ("ragged_b127", 127, 25, 512, 2048, 2350, lambda p: p["nMB"] == 1),
    ("ragged_b129", 129, 25, 512, 2048, 2350, lambda p: p["nMB"] == 2),
    ("tiny_vocab", 640, 25, 384, 1024, 6, lambda p: p["Vp"] == 8 and p["p5_tiles"] == p["nEB"] * (1024 // 128 + 1)),
]


@pytest.mark.parametrize("name,B,L,E,K,V,prop", SHAPES, ids=[c[0] for c in SHAPES])
def test_fused_branch_vs_fp64_chain(cv, name, B, L, E, K, V, prop):
    inp = F.random_inputs(100 + B + K, B, E, K, V, L)
    g, d, sn, r = run_case(cv, name, inp, prop=prop)
    if B == 1:
        # one pair: the loss is identically 0, so are the entropies and every gradient; the accuracies are 1.
        # Bound: the fp32 rounding of exp(S - lse), 1e-6 of w |t| (measured: exactly 0)
        o = sn["out5"].cpu().numpy()
        g.true("B=1 accuracies 1", o[1] == 1.0 and o[2] == 1.0, o[:5].tolist())
        g.le("B=1 |loss| + |entropies|", abs(o[0]) + abs(o[3]) + abs(o[4]), 1e-6)            # [0]
        w = math.exp(S_DEFAULT) * 0.5
        for key, pos in (("du16", sn["txt16"]), ("dm16", sn["img16"])):
            bound = w * float(pos.double().abs().max()) * float(sn["invn"].double().max())
            g.le("B=1 %s / (w |t| invn)" % key, float(sn[key].double().abs().max()) / bound, 1e-6)   # [0]
    g.finish()


def test_fused_long_utterances(cv):
    """L = 77: the second and third 32-position chunks of the text encoder and of the count matrix (whose later
    chunks add to the counts of the earlier ones)."""
    inp = F.long_inputs(384, 512, 2048, 2350, L=77)
    C = F.counts(inp["ids"], 2350)
    early = F.counts(inp["ids"][:, :32], 2350)
    assert ((C > early) & (early > 0)).sum() > 1000        # tokens that repeat across chunks
    g, *_ = run_case(cv, "long_l77", inp)
    g.finish()


def test_fused_natural_two_tiles(cv):
    """T = 2 chosen by the plan, not forced: the largest batch it takes (1536 on 148 SMs), where the head split is
    uneven (11/11/10 of 32 chunks) and P4's warp-per-row schedule wraps around the grid."""
    B = natural_t2_batch(cv)
    inp = F.random_inputs(77, B, 512, 2048, 2350)
    g, *_ = run_case(cv, "natural_t2_b%d" % B, inp,
                     prop=lambda p: p["T"] == 2 and p["KS"] > 1 and p["num_kc"] % p["KS"] != 0 and p["wrapped"])
    g.finish()


def test_fused_unnormalized(cv):
    inp = F.random_inputs(55, 256, 128, 576, 2350)
    inp["table"] *= 0.05
    g, *_ = run_case(cv, "unnormalized", inp, s=0.0, normalize=False, prop=lambda p: p["dw_bn"] == 64)
    g.finish()


@pytest.mark.parametrize("s", [0.0, math.log(100.0)], ids=["s0", "log100"])
def test_fused_device_side_scale(cv, s):
    inp = F.random_inputs(66, 512, 512, 2048, 2350)
    g, *_ = run_case(cv, "device_s_%g" % s, inp, s=s, s_dev=True)
    g.finish()


def test_fused_confident_pairs_and_duplicates(cv):
    """the regime a trained model reaches: P_ii from ~0.3 to ~0.995, plus exact duplicate pairs whose tie is
    decided at each merge level (first index wins, as torch.argmax)."""
    B = 512
    inp = F.aligned_inputs(B)
    # the builders' promises, on the device's own features (the kernel's bf16 features)
    g, d, sn, r = run_case(cv, "confident_dups", inp)
    P = torch.softmax(r["S"], 1).diagonal().cpu().numpy()
    g.values["P_ii min/mean/max"] = [float(P[:-6].min()), float(P.mean()), float(P[:-6].max())]
    g.true("P_ii spread", P[:-6].min() < 0.5 and P.max() > 0.99, g.values["P_ii min/mean/max"])
    for lvl, (i, j) in inp["dups"].items():
        g.true("dup %s: features bit-equal" % lvl, torch.equal(sn["img16"][i], sn["img16"][j])
               and torch.equal(sn["txt16"][i], sn["txt16"][j]))
    # end to end against the fp64 oracle fed the same bf16 operands
    ref = O.contrastive_step(d["x16"].double().cpu(), torch.from_numpy(inp["ids"]), torch.from_numpy(inp["lens"]),
                             d["w16"].double().cpu(), torch.from_numpy(inp["b"]).double(),
                             torch.from_numpy(inp["table"]).double(), S_DEFAULT, "flat", dtype=torch.float64,
                             feature_round="bf16")
    for key, got, want in (("dW", sn["dW"], ref["dW"]), ("db", sn["db"], ref["db"]), ("dtable", sn["dtable"], ref["dtable"])):
        got = got.double().cpu().numpy(); want = want.numpy()
        g.values["e2e %s cos" % key] = c = cosine(got, want)
        g.values["e2e %s rel_fro" % key] = rf = rel_fro(got, want)
        g.true("e2e %s north-star gate" % key, c >= 0.999 and rf <= 2e-2, (c, rf))
    tok = 4 + np.arange(B)
    # measured 3.3e-2 (1.3e-1 with the diagonal of G in bf16): 2x, not 4x, so that the gate keeps that apart
    g.le("e2e dtable worst pair row", F.worst_row(sn["dtable"].cpu()[tok], ref["dtable"][tok]), 6.5e-2)
    g.le("e2e loss rel", abs(float(sn["out5"][0]) - float(ref["loss"])) / float(ref["loss"]), 1e-4)
    for k, key in ((1, "image_accuracy"), (2, "text_accuracy")):
        g.values["e2e %s" % key] = (float(sn["out5"][k]), float(ref[key]))
    g.finish()


def test_token_counts_above_256(cv):
    """one utterance repeats a token 257 times (L = 260): bf16 holds integers exactly only up to 256, so the plan
    sends L > 256 to the multi-kernel step.  Checked through the op, whichever path it takes: d table[v] must be
    257 d table[u] for the token u that utterance holds once, and the step must pass the gate against fp64."""
    import ctypes
    B, E, K, V = 128, 512, 2048, 2350
    inp = F.count257_inputs(B, E, K, V)
    assert F.counts(inp["ids"], V)[0, inp["tok_v"]] == 257
    d = F.device_inputs(inp, DEV)
    g = Gates("counts_257")
    lib = cv._cabi.load()
    g.true("plan rejects L = 260", not lib.cvcl_flat_fused_supported(B, 260, E, K, V))
    g.true("plan takes L = 256", bool(lib.cvcl_flat_fused_supported(B, 256, E, K, V)))
    if not lib.cvcl_flat_fused_supported(B, 260, E, K, V):
        # a direct call returns an error code and runs nothing
        f32 = dict(dtype=torch.float32, device=DEV)
        out5 = torch.full((8,), 7.0, **f32)
        flat = torch.zeros(4 + E + V * E + E * K, **f32)
        ws = torch.zeros(1 << 20, dtype=torch.uint8, device=DEV)
        p = cv.ops._p
        ds, db, dt, dW = cv.ops.split_flat_grads(flat, E, K, V)
        rc = lib.cvcl_flat_step_fused(p(d["x16"]), p(d["w16"]), p(d["ids"]), p(d["lens"]), p(d["b"]), p(d["table"]),
                                      B, 260, E, K, V, 1, S_DEFAULT, None, 1, p(ws), p(out5), None, None, p(dW), p(db),
                                      p(dt), p(ds), None, 0, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        g.true("direct call at L = 260 returns an error", rc != 0, rc)
        g.true("direct call ran nothing", bool((out5 == 7.0).all()) and not bool(flat.any()))
    W = d["w16"].float().requires_grad_(True); b = d["b"].clone().requires_grad_(True)
    table = d["table"].clone().requires_grad_(True)
    out = cv.ops.flat_contrastive_loss(d["x16"].float(), d["ids"], d["lens"], W, b, table, S_DEFAULT, True)
    out[0].backward()
    torch.cuda.synchronize()
    dt = table.grad.double()
    v, u = inp["tok_v"], inp["tok_u"]
    g.le("dtable[v] vs 257 dtable[u]", F.worst_row(dt[v:v + 1], 257.0 * dt[u:u + 1]), 8e-6)          # [1.8e-6]
    ref = O.contrastive_step(d["x16"].double().cpu(), torch.from_numpy(inp["ids"]), torch.from_numpy(inp["lens"]),
                             d["w16"].double().cpu(), torch.from_numpy(inp["b"]).double(),
                             torch.from_numpy(inp["table"]).double(), S_DEFAULT, "flat", dtype=torch.float64,
                             feature_round="bf16")
    g.le("loss rel", abs(out[0].item() - float(ref["loss"])) / float(ref["loss"]), 1e-3)
    for key, got, want in (("dW", W.grad, ref["dW"]), ("dtable", table.grad, ref["dtable"])):
        got = got.double().cpu().numpy(); want = want.numpy()
        c, rf = cosine(got, want), rel_fro(got, want)
        g.true("%s north-star gate" % key, c >= 0.999 and rf <= 2e-2, (c, rf))
    g.le("dtable[v] vs fp64", F.worst_row(dt[v:v + 1].cpu(), ref["dtable"][v:v + 1]), 1e-3)          # [2.2e-4]
    g.finish()
