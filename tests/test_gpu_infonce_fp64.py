"""Every InfoNCE backward outside the one-kernel step, stage by stage against the fp64 chain of tests/_infonce_fp64.py
(fp64 from the kernel's own output of the stage before), in the confident-softmax regime a trained model reaches
(the temperature is trained, so P_ii -> 1) and at the edges of each path:

  a. the multi-kernel flat step cvcl_flat_contrastive_step, every block read from the workspace of ONE full launch
     (ops.flat_step_layout; the step uses atomics, so launches stopped at different phases would not agree);
  b. the feature-level op ops.sim_infonce_fwd / _bwd on one device: the cluster-epilogue form below 4096 pairs and
     the GEMM + addcmul form from 4096 up, after the one-pass and the two-pass forward;
  c. the same op as the ranks of a sharded batch emulated on one device (row block G0 and column block G1, the
     split-K feature gradient at a global batch >= 1536), and the sharded fallback of ops.flat_step_sharded;
  d. the spatial-max InfoNCE backward from a materialised match matrix, square and in row / column blocks.

When a pair is confident, w (P_row,ii + P_col,ii) and -2w nearly cancel: the diagonal of G must enter the feature
gradient in fp32 (gdiag = G_ii - bf16(Gs_ii)), or the bf16 rounding of Gs_ii is left as the whole gradient of that
row.  At one pair the exact loss and gradients are 0: the flat steps give exactly 0; the feature-level op is left
with the rounding of its forward's LSEs.

Each case first asserts the branch it exists to cover.  The committed gates are about 4x the worst errors measured
on a B200; DESIGN section 4 lists both.  Set INFONCE_FP64_REPORT=<file> to append every case's measured values to
<file> as JSON lines."""
import math

import numpy as np
import pytest
import torch

import _fused_fp64 as F
import _infonce_fp64 as N
from _util import O, S_DEFAULT, cosine, rel_fro

pytestmark = pytest.mark.gpu
DEV = "cuda"
D = torch.float64

GATE = dict(                # measured maximum over the cases on a B200 (1000 W) in brackets
    feat_ulp=4.0,           # img16 / txt16 vs fp64 features, bf16 ulps (floor 2^-20 of the row max)    [0.97]
    feat_abs=4e-6,          # fp32 features max abs                                                     [9.7e-7]
    invn_rel=6e-6,          #                                                                           [1.5e-6]
    lse_rel=6e-6,           # both LSE arrays, |error| / max |S|                                        [1.4e-6]
    loss_rel=7e-7,          # |loss error| / max |S| (a confident batch's loss is near 0)               [1.7e-7]
    ent_abs=2.4e-5,         #                                                                           [5.5e-6]
    gs_ulp=1.0,             # Gs vs w (P_row + P_col) from the kernel's LSEs, bf16 ulps                 [0.502]
    gdiag_w=5e-4,           # |gdiag - (G_ii - bf16 Gs_ii)| / w                                         [1.2e-4]
    acc_ulp=72.0,           # feature gradients vs the chain from the kernel's Gs and gdiag, in fp32    [18.6]
                            # ulps of the row's largest |Gs| |K| + |gdiag| |K| (bf16 out: >= 1 bf16 ulp)
    acc_ulp_gemm=900.0,     # the same for the GEMM + addcmul form (contraction 4096 .. 8192)           [220]
    ds_rel=2e-6,            # |ds - ref| / sum |G| |S|                                                  [5.2e-7]
    db_rel=2e-5,            # |db - ref| / sum_r |du_r|                                                 [5.0e-6]
    dw_row=9e-6,            # dW vs du16^T x, worst row                                                 [2.2e-6]
    dt_row=8e-6,            # d table vs C^T dm, worst row                                              [1.9e-6]
    e2e_dw_row=1.5e-2,      # dW against the fp64 oracle, worst row                                     [3.7e-3]
    e2e_big_row=0.5,        # feature gradient against fp64 from 4096 pairs up, worst row               [0.125]
    one_pair=3.2e-6,        # B = 1 through the feature-level op: max |dI| / (w max |feature|)          [8.0e-7]
    match_row=8e-7,         # spatial-max dmatch vs exp(s) G from the kernel's LSEs, worst row        [2.0e-7]
    match_e2e_row=2.1e-4,   # spatial-max dmatch vs fp64 exp(s) G, worst row                            [5.3e-5]
)
NEAR_TIE = 1e-6             # DESIGN section 4: an fp64 top-two gap below 1e-6 max|S| may go either way


def Gates(name):
    return F.Gates(name, "INFONCE_FP64_REPORT")


@pytest.fixture(scope="module")
def cv():
    import multimodal_baby_b200 as m
    m._cabi.load()
    return m


def ulps(got, ref):
    """max |got - ref| in bf16 ulps of ref, with a floor of 2^-20 of each row's max"""
    ref = ref.double(); got = got.double()
    floor = 2.0 ** -20 * ref.abs().amax(1, keepdim=True).clamp_min(1e-300)
    return float(((got - ref).abs() / torch.maximum(F.bf16_ulp(ref), floor)).max())


def acc_ulps(got, ref, mag, bf16_out=False):
    """max |got - ref| in fp32 ulps of each row's largest accumulated magnitude `mag` (the sum of |terms|), and at
    least one bf16 ulp of ref for a bf16 output: what an fp32 accumulation of Gs K + gdiag o K may leave"""
    unit = 2.0 ** -24 * mag.double().amax(1, keepdim=True).clamp_min(1e-300)
    if bf16_out:
        unit = torch.maximum(unit, F.bf16_ulp(ref.double()))
    return float(((got.double() - ref.double()).abs() / unit).max())


def magnitudes(Gs, gd, K):
    """|Gs| |K| + |gdiag| o |K|: the sum of absolute terms of Gs K + gdiag o K"""
    return Gs.double().abs() @ K.double().abs() + gd.double().abs()[:, None] * K.double().abs()


def check_accuracy(g, S, acc, B):
    """the kernel's accuracies (fractions of B) within the fp64 bounds of the near-tie rule"""
    nb = F.accuracy_bounds(S, -(-B // 128), NEAR_TIE).sum(1)
    for z in range(2):
        c = int(round(float(acc[z]) * B))
        g.true("accuracy %d exact up to near-ties" % z, nb[z, 0] <= c <= nb[z, 0] + nb[z, 1],
               "kernel %d ref(sure, near) %s" % (c, nb[z].tolist()))


def check_infonce(g, r, out5, lse, B):
    """LSEs, loss, entropies and accuracies of one device's forward against fp64 on the kernel's features"""
    smax = float(r["S"].abs().max())
    g.le("lse0 max abs / max|S|", (lse[0].double() - r["lse0"]).abs().max() / smax, GATE["lse_rel"])
    g.le("lse1 max abs / max|S|", (lse[1].double() - r["lse1"]).abs().max() / smax, GATE["lse_rel"])
    o = out5.double()
    g.le("loss abs / max|S|", abs(o[0] - r["loss"]) / smax, GATE["loss_rel"])
    g.le("image entropy abs", abs(o[3] - r["ent0"]), GATE["ent_abs"])
    g.le("text entropy abs", abs(o[4] - r["ent1"]), GATE["ent_abs"])
    check_accuracy(g, r["S"], o[1:3], B)


def check_gs(g, r, Gs0, gd0, Gs1=None, gd1=None, w=1.0):
    """Gs within one bf16 ulp of w (P_row + P_col) from the kernel's LSEs, gdiag = G_ii - bf16(Gs_ii) against fp64"""
    g.le("Gs0 ulps", ulps(Gs0, r["Gs64"]), GATE["gs_ulp"])
    g.le("gdiag0 / w", (gd0.double() - r["gdiag"][0]).abs().max() / w, GATE["gdiag_w"])
    if Gs1 is not None:
        g.le("Gs1 ulps", ulps(Gs1, r["Gs64"].t()), GATE["gs_ulp"])
        g.le("gdiag1 / w", (gd1.double() - r["gdiag"][1]).abs().max() / w, GATE["gdiag_w"])


def oracle(d, inp, s, normalize=True):
    return O.contrastive_step(d["x16"].double().cpu(), torch.from_numpy(inp["ids"]), torch.from_numpy(inp["lens"]),
                              d["w16"].double().cpu(), torch.from_numpy(inp["b"]).double(),
                              torch.from_numpy(inp["table"]).double(), s, "flat", normalize=normalize,
                              dtype=torch.float64, feature_round="bf16")


def check_e2e(g, got, ref, pair_rows=None):
    """the step's parameter gradients against the fp64 oracle: north-star gate, and per-row on the confident pairs"""
    for key in ("dW", "db", "dtable"):
        a = got[key].double().cpu().numpy(); b = ref[key].numpy()
        c, rf = cosine(a, b), rel_fro(a, b)
        g.values["e2e %s cos / rel_fro" % key] = (c, rf)
        g.true("e2e %s north-star gate" % key, c >= 0.999 and rf <= 2e-2, (c, rf))
    if pair_rows is not None:
        g.le("e2e dtable worst pair row", F.worst_row(got["dtable"].cpu()[pair_rows], ref["dtable"][pair_rows]),
             N.E2E_WORST_ROW)
    g.le("e2e dW worst row", F.worst_row(got["dW"].cpu(), ref["dW"]), GATE["e2e_dw_row"])


def check_one_pair(g, out5, grads):
    """B = 1: loss, entropies and every feature / parameter gradient exactly 0, accuracies 1"""
    o = out5.cpu().numpy()
    g.true("B=1 accuracies 1", o[1] == 1.0 and o[2] == 1.0, o[:5].tolist())
    g.true("B=1 loss and entropies exactly 0", o[0] == 0 and o[3] == 0 and o[4] == 0, o[:5].tolist())
    for key, t in grads.items():
        g.true("B=1 %s exactly 0" % key, not bool(t.any()), float(t.double().abs().max()))


# ------------------------------------------------------------------------------------------------ a. multi-kernel
def flat_multi(cv, d, s, normalize=True):
    """one full launch of cvcl_flat_contrastive_step -> (outputs, workspace blocks)"""
    from multimodal_baby_b200 import _cabi
    x16, ids, lens = d["x16"], d["ids"], d["lens"]
    B, K = x16.shape; V, E = d["table"].shape; L = ids.shape[1]
    lay = cv.ops.flat_step_layout(B, L, E, K, V)
    ws = torch.zeros(lay["bytes"], dtype=torch.uint8, device=DEV)
    f32 = dict(dtype=torch.float32, device=DEV)
    out5 = torch.zeros(8, **f32)
    img_f = torch.zeros(B, E, **f32); txt_f = torch.zeros(B, E, **f32)
    flat = torch.full((4 + E + V * E + E * K,), float("nan"), **f32)
    ds, db, dtable, dW = cv.ops.split_flat_grads(flat, E, K, V)
    p = cv.ops._p
    _cabi.call("cvcl_flat_contrastive_step", p(x16), 1, p(ids), p(lens), p(d["w16"].float()), p(d["b"]), p(d["table"]),
               B, L, E, K, V, int(normalize), float(s), 1, p(ws), p(out5), p(img_f), p(txt_f), p(dW), p(db), p(dtable),
               p(ds), None, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()

    def blk(name, shape, dtype):
        n = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
        return ws[lay[name]:lay[name] + n].view(dtype).view(*shape).clone()

    sn = dict(out5=out5, img_f=img_f, txt_f=txt_f, ds=ds, db=db, dtable=dtable, dW=dW, flat=flat)
    sn.update(img16=blk("img16", (B, E), torch.bfloat16), txt16=blk("txt16", (B, E), torch.bfloat16),
              invn_i=blk("invn_i", (B,), torch.float32), invn_t=blk("invn_t", (B,), torch.float32),
              lse0=blk("lse0", (B,), torch.float32), lse1=blk("lse1", (B,), torch.float32),
              G0=blk("G0", (B, lay["ldB"]), torch.bfloat16)[:, :B], du16=blk("du16", (B, E), torch.bfloat16),
              dm=blk("dm", (B, E), torch.float32), gdiag=blk("gdiag", (B,), torch.float32))
    return sn


def run_multi(cv, name, inp, s=S_DEFAULT, normalize=True, fused_plan=False):
    """fused_plan: whether the one-kernel plan takes the shape (then FUSED_STEP = False is what sends it here)"""
    g = Gates(name)
    d = F.device_inputs(inp, DEV)
    B, K = d["x16"].shape; V, E = d["table"].shape; L = d["ids"].shape[1]
    assert bool(cv._cabi.load().cvcl_flat_fused_supported(B, L, E, K, V)) == fused_plan, \
        "%s: the one-kernel plan %s this shape" % (name, "rejects" if fused_plan else "takes")
    sn = flat_multi(cv, d, s, normalize)
    scale = math.exp(s); w = scale * 0.5 / B
    # features
    u = d["x16"].double() @ d["w16"].double().t() + d["b"].double()
    inv_i = 1.0 / u.norm(dim=1) if normalize else torch.ones(B, dtype=D, device=DEV)
    img = u * inv_i[:, None]
    txt, inv_t = F.text_features(d["C"], d["table"].double(), d["lens"].double(), normalize)
    g.le("img16 ulps", ulps(sn["img16"], img), GATE["feat_ulp"])
    g.le("txt16 ulps", ulps(sn["txt16"], txt), GATE["feat_ulp"])
    g.le("img_f32 max abs", (sn["img_f"].double() - img).abs().max(), GATE["feat_abs"])
    g.le("txt_f32 max abs", (sn["txt_f"].double() - txt).abs().max(), GATE["feat_abs"])
    g.le("invn_i rel", ((sn["invn_i"].double() - inv_i) / inv_i).abs().max(), GATE["invn_rel"])
    g.le("invn_t rel", ((sn["invn_t"].double() - inv_t) / inv_t).abs().max(), GATE["invn_rel"])
    # similarity, InfoNCE, Gs and the diagonal from the kernel's features and LSEs
    r = N.infonce_chain(sn["img16"], sn["txt16"], s, lse=(sn["lse0"], sn["lse1"]), Gs=sn["G0"], gdiag=sn["gdiag"])
    check_infonce(g, r, sn["out5"], (sn["lse0"], sn["lse1"]), B)
    check_gs(g, r, sn["G0"], sn["gdiag"], w=w)
    g.le("ds rel", F.rel_to(float(sn["ds"][0]) - float(r["ds"]), r["ds_mag"]), GATE["ds_rel"])
    # feature gradients after the normalise backward, from the kernel's Gs, gdiag and inverse norms
    i16, t16 = sn["img16"].double(), sn["txt16"].double()
    lens = d["lens"].double()
    du = N.normalize_bwd(i16, r["dI"], sn["invn_i"].double()) if normalize else r["dI"]
    dm = (N.normalize_bwd(t16, r["dT"], sn["invn_t"].double()) if normalize else r["dT"]) / lens[:, None]
    mag_i = magnitudes(sn["G0"], sn["gdiag"], t16) * sn["invn_i"].double()[:, None]
    mag_t = magnitudes(sn["G0"].t(), sn["gdiag"], i16) * (sn["invn_t"].double() / lens)[:, None]
    g.le("du16 acc ulps", acc_ulps(sn["du16"], du, mag_i, True), GATE["acc_ulp"])
    g.le("dm acc ulps", acc_ulps(sn["dm"], dm, mag_t), GATE["acc_ulp"])
    g.le("db rel", F.rel_to((sn["db"].double() - du.sum(0)).abs().max(), du.abs().sum(0).max()), GATE["db_rel"])
    g.le("dW worst row", F.worst_row(sn["dW"], sn["du16"].double().t() @ d["x16"].double()), GATE["dw_row"])
    present = d["C"].sum(0) > 0
    dt_ref = d["C"].t() @ sn["dm"].double()
    g.le("dtable worst row", F.worst_row(sn["dtable"][present], dt_ref[present]), GATE["dt_row"])
    g.true("dtable absent rows exactly 0", not bool(sn["dtable"][~present].any()))
    g.true("no NaN", not bool(torch.isnan(sn["flat"]).any() or torch.isnan(sn["out5"][:5]).any()))
    return g, d, sn, r


MULTI = [   # name, B, L, E, K, V, builder
    ("e64_golden_shape", 256, 25, 64, 512, 2350, None),
    ("e1024", 256, 25, 1024, 1024, 2350, None),
    ("k1000", 384, 25, 512, 1000, 2350, None),
    ("b2048", 2048, 25, 512, 2048, 2350, None),
    ("l260_counts", 128, 260, 512, 2048, 2350, "count257"),
]


@pytest.mark.parametrize("name,B,L,E,K,V,builder", MULTI, ids=[c[0] for c in MULTI])
def test_multi_kernel_step_off_the_one_kernel_plan(cv, name, B, L, E, K, V, builder):
    inp = F.count257_inputs(B, E, K, V) if builder else F.random_inputs(200 + B + E, B, E, K, V, L)
    g, d, sn, r = run_multi(cv, "multi_" + name, inp)
    g.finish()


@pytest.mark.parametrize("s", [S_DEFAULT, math.log(100.0)], ids=["s_default", "log100"])
def test_multi_kernel_step_confident_pairs(cv, monkeypatch, s):
    """the regime of a trained model at B = 512, with FUSED_STEP = False (the one-kernel plan takes this shape)"""
    monkeypatch.setattr(cv.ops, "FUSED_STEP", False)
    B = 512
    inp = F.aligned_inputs(B)
    assert not cv.ops.fused_supported(B, 25, 512, 2048, B + 4)
    g, d, sn, r = run_multi(cv, "multi_confident_s%.3g" % s, inp, s=s, fused_plan=True)
    P = torch.softmax(r["S"], 1).diagonal()
    g.values["P_ii mean"] = float(P.mean())
    ref = oracle(d, inp, s)
    check_e2e(g, dict(dW=sn["dW"], db=sn["db"], dtable=sn["dtable"]), ref,
              pair_rows=4 + np.arange(B) if s == S_DEFAULT else None)
    g.le("e2e loss rel", abs(float(sn["out5"][0]) - float(ref["loss"])) / float(ref["loss"]), 1e-4)
    g.finish()


@pytest.mark.parametrize("B", [1, 2, 3])
def test_multi_kernel_step_tiny_batches(cv, monkeypatch, B):
    monkeypatch.setattr(cv.ops, "FUSED_STEP", False)
    inp = F.random_inputs(300 + B, B, 512, 2048, 2350)
    g, d, sn, r = run_multi(cv, "multi_b%d" % B, inp, fused_plan=True)
    if B == 1:
        check_one_pair(g, sn["out5"], dict(du16=sn["du16"], dm=sn["dm"], dW=sn["dW"], db=sn["db"],
                                           dtable=sn["dtable"]))
    g.finish()


def test_multi_kernel_step_unnormalized(cv, monkeypatch):
    monkeypatch.setattr(cv.ops, "FUSED_STEP", False)
    inp = F.random_inputs(55, 256, 128, 576, 2350)
    inp["table"] *= 0.05
    g, *_ = run_multi(cv, "multi_unnormalized", inp, s=0.0, normalize=False, fused_plan=True)
    g.finish()


# ------------------------------------------------------------------------------------------------ b. feature level
def confident_features(seed, B, E=512, a_lo=0.4, a_hi=0.8, row_scale=False):
    """unit image rows and text rows txt_i = a_i img_i + sqrt(1 - a_i^2) n_i (n_i unit, orthogonal to img_i);
    row_scale: both multiplied by a per-row factor in [0.5, 2] (pooled rows that are not unit vectors)"""
    gen = torch.Generator().manual_seed(seed)
    img = torch.nn.functional.normalize(torch.randn(B, E, generator=gen, dtype=D), dim=1)
    n = torch.randn(B, E, generator=gen, dtype=D)
    n = torch.nn.functional.normalize(n - (n * img).sum(1, keepdim=True) * img, dim=1)
    a = torch.linspace(a_lo, a_hi, B, dtype=D)[torch.randperm(B, generator=gen)][:, None]
    txt = a * img + (1 - a * a).sqrt() * n
    if row_scale:
        img = img * (0.5 + 1.5 * torch.rand(B, 1, generator=gen, dtype=D))
        txt = txt * (0.5 + 1.5 * torch.rand(B, 1, generator=gen, dtype=D))
    return img.to(DEV).to(torch.bfloat16), txt.to(DEV).to(torch.bfloat16)


def bwd_g(cv, i_q, t_k, t_q, i_k, s, diag_off, coef, lq0, lk0, lq1=None, lk1=None):
    """cvcl_sim_infonce_bwd_g directly -> (Gs0, gdiag0, Gs1 | None, gdiag1 | None)"""
    from multimodal_baby_b200 import _cabi
    p = cv.ops._p
    M0, E = i_q.shape; N0 = t_k.shape[0]
    two = t_q is not None
    M1, N1 = (t_q.shape[0], i_k.shape[0]) if two else (0, 0)
    ld0, ld1 = cv.ops._pad8(N0), cv.ops._pad8(max(N1, 1))
    G0 = torch.empty((M0, ld0), dtype=torch.bfloat16, device=DEV)
    G1 = torch.empty((M1, ld1), dtype=torch.bfloat16, device=DEV) if two else None
    gd0 = torch.empty(M0, dtype=torch.float32, device=DEV)
    gd1 = torch.empty(M1, dtype=torch.float32, device=DEV) if two else None
    ds = torch.zeros(1, dtype=torch.float32, device=DEV)
    _cabi.call("cvcl_sim_infonce_bwd_g", p(i_q), p(t_k), p(t_q), p(i_k), E, M0, N0, M1, N1, E, float(s), int(diag_off),
               float(coef), p(lq0), p(lk0), p(lq1), p(lk1), p(G0), ld0, p(G1), ld1, p(gd0), p(gd1), p(ds),
               torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return G0[:, :N0], gd0, (G1[:, :N1] if two else None), gd1


def one_pass_forward(cv, B, s, unit_norm):
    """the condition under which cvcl_sim_infonce_fwd takes the one-pass similarity (EpiSimStats1P) on one device"""
    return unit_norm and B >= 4096 and B % 256 == 0 and float(np.exp(np.float32(s))) <= 32.0


FEAT = [   # name, B, s, unit rows, one-pass forward, cosines of the pairs
    ("b1", 1, S_DEFAULT, True, False, (0.4, 0.8)),
    ("b2", 2, S_DEFAULT, True, False, (0.4, 0.8)),
    ("b300", 300, S_DEFAULT, True, False, (0.4, 0.8)),
    ("b512", 512, S_DEFAULT, True, False, (0.4, 0.8)),
    ("b512_pooled_rows", 512, S_DEFAULT, False, False, (0.4, 0.8)),
    ("b4096_log32_one_pass", 4096, math.log(32.0), True, True, (0.4, 0.8)),
    ("b8192_log32_one_pass", 8192, math.log(32.0), True, True, (0.4, 0.8)),
    # at exp(s) = 100 a cosine of 0.4 already puts 1 - P_ii below what fp32 LSEs resolve: P_ii ~0.001 .. 1 - 1e-5
    ("b8192_log100_two_pass", 8192, math.log(100.0), True, False, (0.1, 0.3)),
]


@pytest.mark.parametrize("name,B,s,unit,one_pass,cos", FEAT, ids=[c[0] for c in FEAT])
def test_feature_level_op(cv, name, B, s, unit, one_pass, cos):
    g = Gates("feat_" + name)
    assert one_pass_forward(cv, B, s, unit) == one_pass, "%s: not on the forward it covers" % name
    g.values["backward form"] = "gemm+addcmul" if B >= 4096 else "cluster epilogue"
    acc_gate = GATE["acc_ulp_gemm"] if B >= 4096 else GATE["acc_ulp"]
    I, T = confident_features(400 + B, B, a_lo=cos[0], a_hi=cos[1], row_scale=not unit)
    fwd = cv.ops._raw(cv.ops.sim_infonce_fwd); bwd = cv.ops._raw(cv.ops.sim_infonce_bwd)
    out5, l0, l1, a0, a1 = fwd(I, T, T, I, s, 0, 1.0 / B, unit)
    dI, dT, ds = bwd(I, T, T, I, s, 0, 0.5 / B, l0, l1, l1, l0)
    G0, gd0, _, _ = bwd_g(cv, I, T, None, None, s, 0, 0.5 / B, l0, l1)
    torch.cuda.synchronize()
    w = math.exp(s) * 0.5 / B
    r = N.infonce_chain(I, T, s, lse=(l0, l1), Gs=G0, gdiag=gd0)
    check_infonce(g, r, out5, (l0, l1), B)
    check_gs(g, r, G0, gd0, w=w)
    g.le("dI acc ulps vs Gs T + gdiag o T", acc_ulps(dI, r["dI"], magnitudes(G0, gd0, T)), acc_gate)
    g.le("dT acc ulps vs Gs^T I + gdiag o I", acc_ulps(dT, r["dT"], magnitudes(G0.t(), gd0, I)), acc_gate)
    g.le("ds rel", F.rel_to(float(ds[0]) - float(r["ds"]), r["ds_mag"]), GATE["ds_rel"])
    # end to end against the exact fp64 backward on the same bf16 features (unit rows: after the normalise backward,
    # where the diagonal's rounding is not hidden under the component along the row)
    ex = N.infonce_chain(I, T, s, rows_bf16=False)
    one = torch.ones(B, dtype=D, device=DEV)
    proj = (lambda q, x: N.normalize_bwd(q.double(), x.double(), one)) if unit else (lambda q, x: x.double())
    g.values["P_ii mean"] = float(torch.softmax(r["S"], 1).diagonal().mean())
    if B == 1:
        # the exact gradient is 0; what is left is the forward's LSE rounding (lse - S_ii ~1e-7 of exp(s)), not Gs_ii
        o = out5.cpu().numpy()
        g.true("B=1 accuracies 1", o[1] == 1.0 and o[2] == 1.0, o[:5].tolist())
        g.le("B=1 |loss| + |entropies|", abs(o[0]) + abs(o[3]) + abs(o[4]), 2e-6)
        bound = w * float(torch.maximum(I.double().abs().max(), T.double().abs().max()))
        g.le("B=1 max |dI|, |dT| / (w max |feature|)", max(float(dI.abs().max()), float(dT.abs().max())) / bound,
             GATE["one_pair"])
    else:
        e_i = F.worst_row(proj(I, dI), proj(I, ex["dI"])); e_t = F.worst_row(proj(T, dT), proj(T, ex["dT"]))
        lim = N.E2E_WORST_ROW if B < 4096 else GATE["e2e_big_row"]
        g.le("e2e dI worst row", e_i, lim); g.le("e2e dT worst row", e_t, lim)
    g.finish()


# ------------------------------------------------------------------------------------------------ c. sharded
@pytest.mark.parametrize("world,b", [(2, 256), (4, 128), (8, 256)])
def test_emulated_shards_chain(cv, world, b):
    """every rank's row block (G0) and column block (G1) on one GPU, diag_off = r b: together they satisfy the
    one-device chain.  At a global batch >= 1536 the feature gradient splits its contraction over the SMs
    (split-K + featgrad_finish_kernel)."""
    Bg = world * b
    s = S_DEFAULT
    g = Gates("shards_w%d_b%d" % (world, b))
    splitk = Bg >= 1536
    g.values["feature gradient"] = "split-K + featgrad_finish_kernel" if splitk else "cluster epilogue"
    I, T = confident_features(500 + world, Bg)
    fwd = cv.ops._raw(cv.ops.sim_infonce_fwd); bwd = cv.ops._raw(cv.ops.sim_infonce_bwd)
    lse0 = torch.empty(Bg, device=DEV); lse1 = torch.empty(Bg, device=DEV)
    tot = torch.zeros(8, device=DEV)
    for r_ in range(world):
        sl = slice(r_ * b, (r_ + 1) * b)
        out5, l0, l1, _, _ = fwd(I[sl].contiguous(), T, T[sl].contiguous(), I, s, r_ * b, 1.0 / Bg)
        lse0[sl] = l0; lse1[sl] = l1; tot += out5
    dI = torch.empty(Bg, I.shape[1], device=DEV); dT = torch.empty_like(dI); ds = 0.0
    G0 = torch.empty(Bg, Bg, dtype=torch.bfloat16, device=DEV); G1 = torch.empty_like(G0)
    gd0 = torch.empty(Bg, device=DEV); gd1 = torch.empty(Bg, device=DEV)
    for r_ in range(world):
        sl = slice(r_ * b, (r_ + 1) * b)
        iq, tq = I[sl].contiguous(), T[sl].contiguous()
        di, dt, dsr = bwd(iq, T, tq, I, s, r_ * b, 0.5 / Bg, lse0[sl].contiguous(), lse1, lse1[sl].contiguous(), lse0)
        dI[sl] = di; dT[sl] = dt; ds += float(dsr[0])
        G0[sl], gd0[sl], G1[sl], gd1[sl] = bwd_g(cv, iq, T, tq, I, s, r_ * b, 0.5 / Bg, lse0[sl].contiguous(), lse1,
                                                  lse1[sl].contiguous(), lse0)
    w = math.exp(s) * 0.5 / Bg
    r = N.infonce_chain(I, T, s, lse=(lse0, lse1), Gs=(G0, G1), gdiag=(gd0, gd1))
    check_infonce(g, r, tot, (lse0, lse1), Bg)
    check_gs(g, r, G0, gd0, G1, gd1, w=w)
    g.le("dI acc ulps vs chain", acc_ulps(dI, r["dI"], magnitudes(G0, gd0, T)), GATE["acc_ulp"])
    g.le("dT acc ulps vs chain", acc_ulps(dT, r["dT"], magnitudes(G1, gd1, I)), GATE["acc_ulp"])
    g.le("ds rel", F.rel_to(ds - float(r["ds"]), r["ds_mag"]), GATE["ds_rel"])
    ex = N.infonce_chain(I, T, s, rows_bf16=False)
    one = torch.ones(Bg, dtype=D, device=DEV)
    g.le("e2e dI worst row",
         F.worst_row(N.normalize_bwd(I.double(), dI.double(), one), N.normalize_bwd(I.double(), ex["dI"], one)),
         N.E2E_WORST_ROW)
    g.le("e2e dT worst row",
         F.worst_row(N.normalize_bwd(T.double(), dT.double(), one), N.normalize_bwd(T.double(), ex["dT"], one)),
         N.E2E_WORST_ROW)
    g.finish()


@pytest.mark.parametrize("B", [512, 1])
def test_sharded_fallback_one_gpu(cv, B):
    """ops.flat_step_sharded without a group: the fallback orchestration at world 1 (no peer exchange, G1 for the text
    rows, the _ws feature gradient of the image rows)"""
    g = Gates("sharded_fallback_b%d" % B)
    inp = F.aligned_inputs(B) if B > 1 else F.random_inputs(600, 1, 512, 2048, 2350)
    d = F.device_inputs(inp, DEV)
    V, E = d["table"].shape; K = d["x16"].shape[1]
    stats, _, _ = cv.ops.flat_step_sharded(d["x16"], d["ids"], d["lens"], d["w16"].float(), d["b"], d["table"],
                                           S_DEFAULT, True, True, False, None)
    torch.cuda.synchronize()
    ds, db, dtable, dW = cv.ops.split_flat_grads(stats[8:], E, K, V)
    got = dict(dW=dW, db=db, dtable=dtable)
    if B == 1:
        check_one_pair(g, stats[:8], got)
    else:
        ref = oracle(d, inp, S_DEFAULT)
        check_e2e(g, got, ref, pair_rows=4 + np.arange(B))
        g.le("e2e loss rel", abs(float(stats[0]) - float(ref["loss"])) / float(ref["loss"]), 1e-4)
        g.le("e2e ds rel", abs(float(ds[0]) - float(ref["ds"])) / abs(float(ref["ds"])), 1e-3)
    g.finish()


# ------------------------------------------------------------------------------------------------ d. spatial max
def match_reference(match, s, lse=None):
    """fp64 dmatch = exp(s) G of the InfoNCE of logits exp(s) match, G = (P_row + P_col - 2 I) / 2B, from the fp64 LSEs
    or from the kernel's (lse0, lse1); and ds = sum G S with its magnitude sum |G| |S|.  With the kernel's LSEs the
    logits are the kernel's own fp32 products match * fp32(exp(s)): at a confident pair G_ii ~ S_ii - lse is small,
    and the fp32 rounding of exp(s) alone moves it by ~1e-4 relative"""
    if lse is None:
        S = math.exp(s) * match.double()
    else:
        S = (match.float() * float(np.float32(math.exp(float(np.float32(s)))))).double()
    B = S.shape[0]
    l0, l1 = (torch.logsumexp(S, 1), torch.logsumexp(S, 0)) if lse is None else (lse[0].double(), lse[1].double())
    G = torch.exp(S - l0[:, None]) + torch.exp(S - l1[None, :])
    dg = S.diagonal()
    G.diagonal().copy_(torch.expm1(dg - l0) + torch.expm1(dg - l1))
    G *= 0.5 / B
    mag = (G.abs() + torch.eye(B, dtype=D, device=S.device) / B) * S.abs()
    return math.exp(s) * G, (G * S).sum(), mag.sum()


@pytest.mark.parametrize("B", [512, 1])
def test_spatial_max_infonce_backward(cv, B):
    """fp32 throughout (no bf16 Gs): dmatch against exp(s) G from the kernel's own LSEs, where the positive's
    P_row + P_col - 2 cancels when the pair is confident, and against fp64; square and in row / column blocks"""
    g = Gates("match_b%d" % B)
    s = S_DEFAULT
    I, T = confident_features(700 + B, B)
    match = (I.float() @ T.float().t()).contiguous()
    out5, l0, l1, _, _ = cv.ops._raw(cv.ops.match_infonce_fwd)(match, s)
    dmatch, ds = cv.ops._raw(cv.ops.match_infonce_bwd)(match, s, l0, l1)
    dref, ds_ref, ds_mag = match_reference(match, s)
    g.values["P_ii mean"] = float(torch.softmax(math.exp(s) * match.double(), 1).diagonal().mean())
    g.le("dmatch worst row vs chain", F.worst_row(dmatch, match_reference(match, s, (l0, l1))[0]), GATE["match_row"])
    g.le("dmatch worst row vs fp64", F.worst_row(dmatch, dref), GATE["match_e2e_row"])
    g.le("ds rel", F.rel_to(float(ds[0]) - float(ds_ref), ds_mag), GATE["ds_rel"])
    for world in (2, 4) if B > 1 else ():
        b = B // world
        lse0 = torch.empty(B, device=DEV); lse1 = torch.empty(B, device=DEV)
        blocks = []
        for r_ in range(world):
            sl = slice(r_ * b, (r_ + 1) * b)
            mr, mc = match[sl].contiguous(), match[:, sl].contiguous()
            _, a, c, _, _ = cv.ops._raw(cv.ops.match_infonce_block_fwd)(mr, mc, r_ * b, s, 1.0 / B)
            lse0[sl] = a; lse1[sl] = c; blocks.append((mr, mc))
        dr_all = torch.empty(B, B, device=DEV); dc_all = torch.empty(B, B, device=DEV); dsb = 0.0
        for r_, (mr, mc) in enumerate(blocks):
            sl = slice(r_ * b, (r_ + 1) * b)
            dr, dc, dsr = cv.ops._raw(cv.ops.match_infonce_block_bwd)(mr, mc, r_ * b, s, 0.5 / B, lse0[sl].contiguous(),
                                                                      lse1, lse0, lse1[sl].contiguous())
            dr_all[sl] = dr; dc_all[:, sl] = dc; dsb += float(dsr[0])
        dchain = match_reference(match, s, (lse0, lse1))[0]
        g.le("world %d row blocks worst row vs chain" % world, F.worst_row(dr_all, dchain), GATE["match_row"])
        g.le("world %d column blocks worst column vs chain" % world, F.worst_row(dc_all.t(), dchain.t()),
             GATE["match_row"])
        g.le("world %d row blocks worst row vs fp64" % world, F.worst_row(dr_all, dref), GATE["match_e2e_row"])
        g.le("world %d ds rel" % world, F.rel_to(dsb - float(ds_ref), ds_mag), GATE["ds_rel"])
    if B == 1:
        o = out5.cpu().numpy()
        g.true("B=1 loss exactly 0", o[0] == 0, o[:5].tolist())
        g.true("B=1 dmatch and ds exactly 0", not bool(dmatch.any()) and float(ds[0]) == 0.0,
               (float(dmatch.abs().max()), float(ds[0])))
    g.finish()
