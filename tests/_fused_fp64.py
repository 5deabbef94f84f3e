"""fp64 chain reference of the one-kernel flat step (csrc/fused_step.cuh) and the input builders of its edge tests.

Each phase is checked against fp64 computed from the kernel's OWN output of the previous phase (read from the
workspace through ops.fused_layout after a launch with phase_limit = 1..5, then 0).  What is left between the two
is that phase's fp32 accumulation order and the bf16 roundings the kernel documents, so the gates can be orders of
magnitude tighter than a whole-step comparison, and a failure names the phase.

    chain_reference(inp, snap, s)  -- pure torch, any device (float64); CPU tests feed it unrounded values
    capture(cv, d, s, ...)         -- GPU: launch the kernel phase by phase and read the workspace blocks
    random_inputs / aligned_inputs / long_inputs / count257_inputs -- builders (numpy)

Test infrastructure.
"""
import json
import math
import os

import numpy as np
import torch

from _util import O

SOS, EOS = O.SOS_TOKEN_ID, O.EOS_TOKEN_ID


# ------------------------------------------------------------------------------------------------ builders
def bf16_round(a):
    """numpy fp32 -> bf16 -> fp32 (round to nearest even), as torch does."""
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).bfloat16().float().numpy()


def random_inputs(seed, B, E, K, V, L=25):
    rng = np.random.RandomState(seed)
    f = O.synth_trunk_features(rng, (B, K))
    ids, lens = O.synth_tokens(rng, B, L, V)
    W, b, table = O.synth_weights(np.random.RandomState(seed + 1), E, K, V)
    return dict(f=f, ids=ids, lens=lens, W=W, b=b, table=table)


# merge levels of an exact tie between columns i < j (rows of 128, half tiles of 64, chunks of 32 columns):
# same chunk, another chunk of the same half tile, the other half tile, another column block
DUP_LEVELS = {"chunk": (5, 20), "half": (10, 40), "tile": (30, 100), "block": (50, 300)}


def aligned_inputs(B, E=512, K=2048, V=None, L=25, seed=11, a_lo=0.4, a_hi=0.8, n_loose=6, dups=DUP_LEVELS):
    """Confident pairs: pair i is [SOS, tok_i, EOS] with a token of its own (tok_i = 4 + i), and its table row is
    a_i * u_i/|u_i| + sqrt(1 - a_i^2) * n_i (n_i a random unit vector orthogonal to u_i), where u = bf16(x) bf16(W)^T + b
    in fp64.  The text feature of pair i is then that row, its cosine with its image is a_i, and P_ii spans
    ~0.3 .. 0.993 at B = 512, s = -log 0.07.  The last `n_loose` pairs get a_i ~ 0.05: their arg-max is decided
    among unrelated columns, with fp64 near-ties.  `dups` {name: (i, j)}: pair j is a byte copy of pair i (same x row,
    same ids), an exact tie between columns i and j at the named merge level; both get a_i = 0.8."""
    V = V or B + 4
    assert V >= B + 4
    rng = np.random.RandomState(seed)
    f = rng.standard_normal((B, K)).astype(np.float32)      # zero-mean: the image features are nearly orthogonal
    W, b, _ = O.synth_weights(np.random.RandomState(seed + 1), E, K, 8)
    u = bf16_round(f).astype(np.float64) @ bf16_round(W).astype(np.float64).T + b.astype(np.float64)
    uh = u / np.linalg.norm(u, axis=1, keepdims=True)
    a = np.linspace(a_lo, a_hi, B)
    rng.shuffle(a)
    a[B - n_loose:] = rng.uniform(0.0, 0.1, n_loose)
    dups = {k: v for k, v in (dups or {}).items() if v[1] < B}
    for i, j in dups.values():
        a[i] = a[j] = 0.8
    n = rng.standard_normal((B, E))
    n -= (n * uh).sum(1, keepdims=True) * uh
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    table = rng.standard_normal((V, E)).astype(np.float32)
    table[[0, SOS, EOS]] = 0.0
    table[4:4 + B] = (a[:, None] * uh + np.sqrt(1.0 - a[:, None] ** 2) * n).astype(np.float32)
    ids = np.zeros((B, L), np.int64)
    ids[:, 0] = SOS; ids[:, 1] = 4 + np.arange(B); ids[:, 2] = EOS
    lens = np.full(B, 3, np.int64)
    for i, j in dups.values():
        f[j] = f[i]; ids[j] = ids[i]; lens[j] = lens[i]
    return dict(f=f, ids=ids, lens=lens, W=W, b=b, table=table, a=a, dups=dups)


def long_inputs(B, E, K, V, L=77, seed=21):
    """Utterances of 40..L tokens drawn from a pool of 12 tokens per row, so that most tokens repeat across the
    32-position chunks of the text encoder and of the count matrix."""
    rng = np.random.RandomState(seed)
    d = random_inputs(seed, B, E, K, V, 25)
    ids = np.zeros((B, L), np.int64)
    lens = rng.randint(40, L + 1, size=B).astype(np.int64)
    for r in range(B):
        pool = rng.randint(4, V, size=12)
        ids[r, 0] = SOS
        ids[r, 1:lens[r] - 1] = pool[rng.randint(0, 12, size=lens[r] - 2)]
        ids[r, lens[r] - 1] = EOS
    d.update(ids=ids, lens=lens)
    return d


def count257_inputs(B, E, K, V, seed=31):
    """L = 260; pair 0 is [SOS, v x 257, u, EOS] with tokens v and u used nowhere else, the rest are random
    utterances of up to 25 tokens (padded to 260).  d table[v] = 257 d table[u] exactly."""
    d = random_inputs(seed, B, E, K, V, 25)
    v, u = 4, 5
    ids = np.zeros((B, 260), np.int64)
    body = d["ids"]
    body = np.where((body == v) | (body == u), 6, body)
    ids[:, :25] = body
    ids[0] = 0
    ids[0, 0] = SOS; ids[0, 1:258] = v; ids[0, 258] = u; ids[0, 259] = EOS
    lens = d["lens"].copy(); lens[0] = 260
    d.update(ids=ids, lens=lens, tok_v=v, tok_u=u)
    return d


def counts(ids, V):
    """C[b, v] = #{l : ids[b, l] = v}, column 0 (pad) zero -- exact integers (numpy bincount)."""
    B = ids.shape[0]
    C = np.zeros((B, V), np.float64)
    for r in range(B):
        C[r] = np.bincount(ids[r], minlength=V)[:V]
    C[:, 0] = 0
    return C


# ------------------------------------------------------------------------------------------------ reference
class Gates:
    """collects every gate of one case, appends the measured values to the file named by the environment variable
    `report_env` (JSON lines) when it is set, then fails with every gate that did not hold"""
    def __init__(self, name, report_env):
        self.name, self.report_env, self.values, self.failed = name, report_env, {}, []

    def le(self, key, value, limit):
        value = float(value)
        self.values[key] = value
        if not (value <= limit):
            self.failed.append("%s = %.3e > %.1e" % (key, value, limit))

    def true(self, key, cond, info=None):
        self.values[key] = bool(cond) if info is None else info
        if not cond:
            self.failed.append("%s failed (%s)" % (key, info))

    def finish(self):
        path = os.environ.get(self.report_env)
        if path:
            with open(path, "a") as fh:
                fh.write(json.dumps({"case": self.name, **self.values}) + "\n")
        assert not self.failed, "%s: %s" % (self.name, "; ".join(self.failed))


def worst_row(got, ref):
    """max over rows of |got - ref|_2 / |ref|_2 (rows that are zero on both sides count 0)."""
    got = got.double().reshape(got.shape[0], -1); ref = ref.double().reshape(ref.shape[0], -1)
    num = (got - ref).norm(dim=1); den = ref.norm(dim=1)
    r = torch.where(num == 0, torch.zeros_like(num), num / den)
    return float(r.max()) if r.numel() else 0.0


def rel_to(diff, mag):
    """|diff| / mag, 0 when diff is 0 (a scale of 0 then does not matter)"""
    diff, mag = abs(float(diff)), float(mag)
    return 0.0 if diff == 0 else diff / max(mag, 1e-300)


def first_argmax_and_gap(S):
    """per row: first index of the maximum, and the gap between the maximum and the largest value that is NOT
    equal to it (0 < gap < tol is an fp64 near-tie; an exact tie has the first index as its only right answer)."""
    top = S.max(dim=1)
    arg = (S == top.values[:, None]).int().argmax(dim=1)
    rest = torch.where(S == top.values[:, None], torch.full_like(S, -math.inf), S)
    gap = top.values - rest.max(dim=1).values
    return arg, gap


def text_features(C, table, lens, normalize):
    m = (C @ table) / lens[:, None]
    if not normalize:
        return m, torch.ones(m.shape[0], dtype=m.dtype, device=m.device)
    inv = 1.0 / m.norm(dim=1).clamp_min(1e-12)
    return m * inv[:, None], inv


def bf16_ulp(x):
    """one bf16 ulp at |x| (8 significant bits)."""
    ax = x.abs().clamp_min(1e-38)
    return torch.exp2(torch.floor(torch.log2(ax)) - 7)


def chain_reference(inp, snap, s, normalize=True, rows_bf16=True):
    """fp64 reference of every phase from the kernel's own output of the previous phase.

    inp:  x16, w16, b, table, ids, lens, C (float64 counts) -- tensors on one device
    snap: the kernel's blocks: hpart [KS,B,E], img16/txt16 [B,E], img_f/txt_f [B,E], invn [2,B], lse [2,B],
          diag [2,B], gdiag [2,B] (bf16 Gs_ii of P3), dq [2,B,E] (slab sums), du16/dm16 [B,E]
    Returns {name: fp64 tensor}.  rows_bf16=False (host tests, no kernel): bf16 roundings are not applied, so
    the chain equals the exact fp64 step."""
    D = torch.float64
    x, w = inp["x16"].to(D), inp["w16"].to(D)
    b, table, lens, C = inp["b"].to(D), inp["table"].to(D), inp["lens"].to(D), inp["C"].to(D)
    B = x.shape[0]
    scale = math.exp(s)
    wg = scale * 0.5 / B
    r = {}
    # P0 / P1: head, text encoder, normalise
    r["u"] = x @ w.t() + b
    hp = snap["hpart"].to(D).sum(0) + b
    r["invn_i"] = 1.0 / hp.norm(dim=1).clamp_min(1e-12) if normalize else torch.ones(B, dtype=D, device=x.device)
    r["img"] = hp * r["invn_i"][:, None]
    r["txt"], r["invn_t"] = text_features(C, table, lens, normalize)
    # P2 / P3 from the kernel's bf16 features
    img16, txt16 = snap["img16"].to(D), snap["txt16"].to(D)
    S = scale * (img16 @ txt16.t())
    r["S"] = S
    r["lse0"], r["lse1"] = torch.logsumexp(S, 1), torch.logsumexp(S, 0)
    dg = S.diagonal()
    r["diag"] = dg
    P0 = torch.softmax(S, 1); P1 = torch.softmax(S, 0)
    r["loss"] = 0.5 * ((r["lse0"] - dg).mean() + (r["lse1"] - dg).mean())
    r["ent0"] = (r["lse0"] - (P0 * S).sum(1)).mean()
    r["ent1"] = (r["lse1"] - (P1 * S).sum(0)).mean()
    G = wg * (P0 + P1) - 2 * wg * torch.eye(B, dtype=D, device=x.device)
    r["ds"] = (G * (S / scale)).sum()                  # dL/ds = sum (P0 + P1 - 2I) / (2B) * S
    r["ds_mag"] = ((wg * (P0 + P1) + 2 * wg * torch.eye(B, dtype=D, device=x.device)) * (S / scale).abs()).sum()
    # dQ from the kernel's LSEs: Gs = w (P_row + P_col), the bf16 A operand, diagonal included
    lk = snap["lse"].to(D)
    Gs = wg * (torch.exp(S - lk[0][:, None]) + torch.exp(S - lk[1][None, :]))
    r["gdiag"] = Gs.diagonal().clone()                 # P3 records bf16 of this for P4
    if rows_bf16:
        Gs = Gs.to(torch.bfloat16).to(D)
    r["dq0"], r["dq1"] = Gs @ txt16, Gs.t() @ img16
    # P4 from the kernel's dQ sums, invn, diag, LSEs and recorded bf16 Gs_ii: the slabs' Gs_ii K_i is replaced by
    # G_ii K_i, G_ii = w (P_row,ii - 1 + P_col,ii - 1)
    kd, kdq, kinv, kgd = snap["diag"].to(D), snap["dq"].to(D), snap["invn"].to(D), snap["gdiag"].to(D)
    for z, (q, pos) in enumerate(((img16, txt16), (txt16, img16))):
        coef = wg * (torch.expm1(kd[z] - lk[z]) + torch.expm1(kd[z] - lk[1 - z])) - kgd[z]
        acc = kdq[z] + coef[:, None] * pos
        if normalize:
            acc = (acc - q * (q * acc).sum(1, keepdim=True)) * kinv[z][:, None]
        if z == 1:
            acc = acc / lens[:, None]
        r["du" if z == 0 else "dm"] = acc
    r["db"] = r["du"].sum(0)
    r["db_mag"] = r["du"].abs().sum(0)
    # P5 from the kernel's bf16 P4 rows
    du16, dm16 = snap["du16"].to(D), snap["dm16"].to(D)
    r["dW"] = du16.t() @ x
    r["dtable"] = C.t() @ dm16
    return r


def accuracy_bounds(S, nMB, rel_tie=1e-6, excuse=None):
    """per direction and row block: (sure, ties) -- the rows whose first-index fp64 arg-max is the positive and
    whose top-two gap is not an fp64 near-tie, and the number of near-tie rows (0 < gap < rel_tie * max|S|).
    excuse [2, B] (optional): rows counted as near-ties whatever their gap."""
    B = S.shape[0]
    tol = rel_tie * float(S.abs().max())
    out = np.zeros((2, nMB, 2), np.int64)
    for z, Sz in enumerate((S, S.t())):
        arg, gap = first_argmax_and_gap(Sz)
        near = (gap > 0) & (gap < tol)
        if excuse is not None:
            near = near | excuse[z]
        ok = (arg == torch.arange(B, device=S.device)) & ~near
        for rb in range(nMB):
            sl = slice(rb * 128, min(B, rb * 128 + 128))
            out[z, rb, 0] = int(ok[sl].sum()); out[z, rb, 1] = int(near[sl].sum())
    return out


# ------------------------------------------------------------------------------------------------ GPU capture
def plan(lay, B, E, K, V):
    """the plan properties the edge cases exist to cover, from ops.fused_layout."""
    nEB = E // 128
    T = lay["nCB"] // lay["nPart"]
    n_p5 = nEB * (K // lay["dw_bn"]) + -(-V // 128) * nEB
    return dict(T=T, KS=lay["KS"], QS=lay["QS"], nEB=nEB, dw_bn=lay["dw_bn"], Vp=lay["Vp"], grid=lay["grid"],
                nMB=lay["Bp"] // 128, p5_tiles=n_p5, num_kc=K // 64, wrapped=2 * B > lay["grid"] * 8)


def device_inputs(inp, dev):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)   # noqa: E731
    d = dict(x16=t(inp["f"]).bfloat16().contiguous(), w16=t(inp["W"]).bfloat16().contiguous(), b=t(inp["b"]),
             table=t(inp["table"]), ids=t(inp["ids"]), lens=t(inp["lens"]))
    d["C"] = t(counts(inp["ids"], inp["table"].shape[0]))
    return d


def capture(cv, d, s, normalize=True, s_dev=None, replays=5):
    """run cvcl_flat_step_fused with phase_limit = 1..5 and 0, read each phase's blocks right after it, then
    replay the whole step `replays` times.  s_dev: a CUDA scalar read by the kernel (the host s is then NaN)."""
    from multimodal_baby_b200 import _cabi
    x16, w16, ids, lens = d["x16"], d["w16"], d["ids"], d["lens"]
    B, K = x16.shape; V, E = d["table"].shape; L = ids.shape[1]
    lay = cv.ops.fused_layout(B, L, E, K, V)
    Bp, KS, nPart, nCB, Vp = lay["Bp"], lay["KS"], lay["nPart"], lay["nCB"], lay["Vp"]
    dev = x16.device
    ws = torch.zeros(lay["bytes"], dtype=torch.uint8, device=dev)
    f32 = dict(dtype=torch.float32, device=dev)
    out5 = torch.zeros(8, **f32)
    img_f = torch.zeros(B, E, **f32); txt_f = torch.zeros(B, E, **f32)
    flat = torch.full((4 + E + V * E + E * K,), float("nan"), **f32)
    ds, db, dtable, dW = cv.ops.split_flat_grads(flat, E, K, V)
    p = cv.ops._p
    st = torch.cuda.current_stream().cuda_stream
    host_s = float("nan") if s_dev is not None else s

    def launch(limit):
        _cabi.call("cvcl_flat_step_fused", p(x16), p(w16), p(ids), p(lens), p(d["b"]), p(d["table"]), B, L, E, K, V,
                   int(normalize), host_s, p(s_dev), 1, p(ws), p(out5), p(img_f), p(txt_f), p(dW), p(db), p(dtable),
                   p(ds), None, limit, st)
        torch.cuda.synchronize()

    def blk(name, n, dtype):
        nbytes = n * torch.empty(0, dtype=dtype).element_size()
        return ws[lay[name]:lay[name] + nbytes].view(dtype)

    sn = {}
    launch(1)
    sn["hpart"] = blk("hpart", KS * Bp * E, torch.float32).view(KS, Bp, E)[:, :B].clone()
    sn["txt16"] = blk("txt16", Bp * E, torch.bfloat16).view(Bp, E)[:B].clone()
    sn["txt_f"] = txt_f.clone()
    sn["invn_t"] = blk("invn", 2 * Bp, torch.float32).view(2, Bp)[1, :B].clone()
    launch(2)
    sn["img16"] = blk("img16", Bp * E, torch.bfloat16).view(Bp, E)[:B].clone()
    sn["img_f"] = img_f.clone()
    sn["invn"] = blk("invn", 2 * Bp, torch.float32).view(2, Bp)[:, :B].clone()
    sn["cmat"] = blk("cmat", Bp * Vp, torch.bfloat16).view(Bp, Vp)[:B, :V].clone()
    launch(3)
    part = blk("part", 2 * 2 * nCB * Bp * 4, torch.float32).view(2, 2 * nCB, Bp, 4)[:, :, :B]
    sn["part_m"] = part[..., 0].clone()
    sn["part_arg"] = blk("part", 2 * 2 * nCB * Bp * 4, torch.int32).view(2, 2 * nCB, Bp, 4)[:, :, :B, 3].clone()
    sn["diag"] = blk("diag", 2 * Bp, torch.float32).view(2, Bp)[:, :B].clone()
    launch(4)
    sn["lse"] = blk("lse", 2 * Bp, torch.float32).view(2, Bp)[:, :B].clone()
    sn["gdiag"] = blk("gdiag", 2 * Bp, torch.float32).view(2, Bp)[:, :B].clone()
    sn["dq"] = blk("dqpart", 2 * nPart * Bp * E, torch.float32).view(2, nPart, Bp, E)[:, :, :B].double().sum(1)
    sn["rb_part"] = blk("rb_part", 2 * (Bp // 128) * 6, torch.float32).view(2, Bp // 128, 6).clone()
    launch(5)
    sn["du16"] = blk("du16", Bp * E, torch.bfloat16).view(Bp, E)[:B].clone()
    sn["dm16"] = blk("dm16", Bp * E, torch.bfloat16).view(Bp, E)[:B].clone()
    flat.fill_(float("nan")); out5.zero_()
    launch(0)
    sn["out5"] = out5.clone(); sn["flat"] = flat.clone()
    sn["ds"], sn["db"], sn["dtable"], sn["dW"] = (t.clone() for t in cv.ops.split_flat_grads(sn["flat"], E, K, V))
    same = True
    for _ in range(replays):
        launch(0)
        same = same and torch.equal(out5[:5], sn["out5"][:5]) and torch.equal(flat[:1], sn["flat"][:1]) \
            and torch.equal(flat[4:], sn["flat"][4:])
    sn["replays_identical"] = same
    sn["ctrl"] = ws[:16].view(torch.int32).cpu().tolist()
    sn["lay"] = lay
    return sn


def sharded_world1(cv, d, s, normalize=True):
    """cvcl_flat_step_fused_sharded at world 1 (the sharded instance, peer tables naming local buffers)
    -> (out5, flat gradient buffer)."""
    import ctypes
    from multimodal_baby_b200 import _cabi
    x16, w16, ids, lens = d["x16"], d["w16"], d["ids"], d["lens"]
    B, K = x16.shape; V, E = d["table"].shape; L = ids.shape[1]
    dev = x16.device
    lib = _cabi.load()
    p = cv.ops._p
    f32 = dict(dtype=torch.float32, device=dev)
    out5 = torch.zeros(8, **f32)
    flat = torch.zeros(4 + E + V * E + E * K, **f32)
    ds, db, dt, dW = cv.ops.split_flat_grads(flat, E, K, V)
    ws = torch.zeros(int(lib.cvcl_flat_fused_sharded_workspace_bytes(B, L, E, K, V, 1)), dtype=torch.uint8, device=dev)
    txt_all = torch.zeros(B, E, dtype=torch.bfloat16, device=dev); img_all = torch.zeros_like(txt_all)
    part_all = torch.zeros(int(lib.cvcl_flat_fused_sharded_part_bytes(B, 1)) // 4, **f32)
    flags = torch.zeros(32, dtype=torch.int32, device=dev); epoch = torch.zeros(1, dtype=torch.int32, device=dev)
    arr = ctypes.c_void_p * 1
    _cabi.call("cvcl_flat_step_fused_sharded", p(x16), p(w16), p(ids), p(lens), p(d["b"]), p(d["table"]),
               B, L, E, K, V, int(normalize), s, None, 1, p(ws), p(out5), None, None, p(dW), p(db), p(dt), p(ds), None, 0,
               1, 0, arr(txt_all.data_ptr()), arr(img_all.data_ptr()), arr(part_all.data_ptr()), arr(flags.data_ptr()),
               epoch.data_ptr(), None, None, 0, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return out5, flat
