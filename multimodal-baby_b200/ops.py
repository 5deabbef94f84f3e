"""torch.library custom ops over the C ABI of libcvcl_b200.so + their autograd wiring.

Every op in the `cvcl_b200::` namespace is a thin marshalling layer: it allocates the outputs
with torch (torch owns all device memory), passes raw device pointers, sizes and the current
CUDA stream to one `extern "C"` entry point, and returns.  There is NO CPU implementation:
CPU tensors raise, and a missing shared library raises `CvclLibraryMissing` at first use.

Reference call sites replaced (paths relative to the reference repo):
  text_features     multimodal/multimodal.py:496-503, 575-584, 743
  head_features     multimodal/multimodal.py:181-192 (applied at :101), 736
  sim_logits        multimodal/multimodal.py:755, 783-794
  sim_infonce       multimodal/multimodal.py:755, 783-787, 801-818 (+ autograd)
  spatial_max_infonce     multimodal/multimodal.py:771-822 with the batch sharded over a process group
  flat_contrastive_step   multimodal/multimodal.py:796-822 + loss.backward()
  eval_nway         multimodal/multimodal_lit.py:466-511, eval.py:196-214
  conv1x1_f32, eval_nway_spatial, classify_ncat_spatial
                    the same evaluation for spatial embeddings (multimodal/multimodal.py:181-185, 757-787)
  spatial_attention_f32
                    the per-location terms of the spatial similarity, before its reductions (multimodal/multimodal.py:771-780)
  retrieval_f32     image->text / text->image retrieval (top-K, rank of the first positive, recall@K) on the
                    evaluation scores above
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _cabi

_NS = "cvcl_b200"


# ----------------------------------------------------------------------------------------
# marshalling helpers
# ----------------------------------------------------------------------------------------
def _p(t: Optional[Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    """raw handle of the current CUDA stream (the C-level query: torch.cuda.current_stream() builds a Stream object
    and costs ~6 us per call, this ~0.3 us)"""
    return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("cvcl_b200 ops run only on CUDA (sm_100a) tensors; there is no CPU "
                               "fallback (got a %s tensor)" % t.device)


_TOKEN_STATUS = {}


def token_status(dev) -> Tensor:
    """persistent int32 word per device: the text-encoder kernels set it to 1 when they meet a token id outside
    [0, V) (they then treat the id as <pad>; the reference's nn.Embedding fails with a device-side assert)."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    t = _TOKEN_STATUS.get(key)
    if t is None:
        t = _TOKEN_STATUS[key] = torch.zeros((1,), dtype=torch.int32, device=dev)
    return t


def check_token_ids(dev=None):
    """Raise IndexError if any text-encoder launch since the last check saw a token id outside the embedding table
    (a vocabulary / checkpoint mismatch would otherwise train silently on <pad> rows).  Synchronises: call it where
    a sync is acceptable (epoch end, validation, or once per dataset)."""
    items = list(_TOKEN_STATUS.items()) if dev is None else \
        [(k, v) for k, v in _TOKEN_STATUS.items() if k == (dev.index if dev.index is not None else torch.cuda.current_device())]
    for _, t in items:
        if int(t.item()) != 0:
            t.zero_()
            raise IndexError("cvcl_b200: a token id outside [0, vocab_size) reached the text encoder")


def _scalar(s) -> float:
    """host value of the log-scale `s` (a python float, a CPU 0-dim tensor when the temperature is
    fixed -- multimodal.py:712 -- or a CUDA Parameter, in which case this is the one D2H sync the
    reference's own logging already performs every step, multimodal_lit.py:252)."""
    return float(s.detach()) if torch.is_tensor(s) else float(s)


def _raw(op):
    """The python body of a torch.library custom op.  The ops stay registered (`cvcl_b200::*`: schema,
    fake kernels, traceability); the eager autograd wrappers below call the body directly because the
    dispatcher round trip costs ~40 us per call, which is a third of the whole B=512 step."""
    return getattr(op, "_init_fn", op)


def _pad8(n: int) -> int:
    return (n + 7) // 8 * 8


def _i64(t: Tensor) -> Tensor:
    if t.dtype != torch.int64:
        raise TypeError("token ids / lengths must be int64 (got %s)" % t.dtype)
    return t if t.is_contiguous() else t.contiguous()


def _f32(t: Tensor) -> Tensor:
    if t.dtype == torch.float32 and t.is_contiguous():
        return t.detach() if t.requires_grad else t
    return t.detach().to(torch.float32).contiguous()


def to_bf16_pair(x: Tensor, want_t: bool) -> Tuple[Tensor, Optional[Tensor]]:
    """[R,C] fp32/bf16 -> (bf16 [R,C] contiguous, bf16 transposed [C, pad8(R)] or None)."""
    x = x.detach()
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    x = x.contiguous()
    R, C = x.shape
    if x.dtype == torch.bfloat16 and not want_t:
        return x, None
    dst = x if x.dtype == torch.bfloat16 else torch.empty((R, C), dtype=torch.bfloat16, device=x.device)
    ldt = _pad8(R)
    dst_t = torch.empty((C, ldt), dtype=torch.bfloat16, device=x.device) if want_t else None
    _cabi.call("cvcl_cast_transpose", _p(x), int(x.dtype == torch.bfloat16),
               None if dst is x else _p(dst), _p(dst_t), 1, R, C, C, C, ldt, 0, 0, 0, _stream())
    return dst, dst_t


# ----------------------------------------------------------------------------------------
# K1 text encoder
# ----------------------------------------------------------------------------------------
@torch.library.custom_op(_NS + "::text_encoder_fwd", mutates_args=())
def text_encoder_fwd(ids: Tensor, lens: Tensor, table: Tensor, normalize: bool, per_token: bool,
                     pool_scale: float, want_tok: bool = True) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (feat [B,E] fp32, inv_norm [B] or [B*L] fp32, tok [B,L,E] fp32 (per_token and want_tok) or empty).
    want_tok=False (spatial "mean" similarity, which only consumes the pooled factor) skips the
    [B,L,E] per-token output."""
    _need_cuda(ids, lens, table)
    ids = _i64(ids); lens = _i64(lens); table = _f32(table)
    B, L = ids.shape
    V, E = table.shape
    dev = ids.device
    feat = torch.empty((B, E), dtype=torch.float32, device=dev)
    inv = torch.empty((B * L if per_token else B,), dtype=torch.float32, device=dev)
    tok = torch.empty((B, L, E) if (per_token and want_tok) else (0,), dtype=torch.float32, device=dev)
    _cabi.call("cvcl_text_encoder_fwd", _p(ids), _p(lens), _p(table), B, L, E, V, int(normalize),
               int(per_token), float(pool_scale), _p(feat), None, 0, _p(inv),
               _p(tok) if (per_token and want_tok) else None, None, _p(token_status(dev)), _stream())
    return feat, inv, tok


@text_encoder_fwd.register_fake
def _(ids, lens, table, normalize, per_token, pool_scale, want_tok=True):
    B, L = ids.shape
    E = table.shape[1]
    return (table.new_empty((B, E)), table.new_empty((B * L if per_token else B,)),
            table.new_empty((B, L, E) if (per_token and want_tok) else (0,)))


@torch.library.custom_op(_NS + "::embedding_bag_bwd", mutates_args=())
def embedding_bag_bwd(ids: Tensor, lens: Tensor, g: Tensor, feat: Tensor, inv_norm: Tensor,
                      normalize: bool, V: int) -> Tensor:
    _need_cuda(ids, g)
    ids = _i64(ids); lens = _i64(lens); g = _f32(g)
    B, L = ids.shape
    E = g.shape[1]
    dtable = torch.zeros((V, E), dtype=torch.float32, device=g.device)
    _cabi.call("cvcl_embedding_bag_bwd", _p(ids), _p(lens), _p(g), _p(feat.contiguous()),
               _p(inv_norm), int(normalize), _p(dtable), B, L, E, V, _stream())
    return dtable


@embedding_bag_bwd.register_fake
def _(ids, lens, g, feat, inv_norm, normalize, V):
    return g.new_empty((V, g.shape[1]))


@torch.library.custom_op(_NS + "::text_token_bwd", mutates_args=())
def text_token_bwd(ids: Tensor, lens: Tensor, table: Tensor, dtok: Optional[Tensor],
                   dpool: Optional[Tensor], pool_scale: float, normalize: bool) -> Tensor:
    _need_cuda(ids, table)
    ids = _i64(ids); lens = _i64(lens); table = _f32(table)
    B, L = ids.shape
    V, E = table.shape
    dtok = None if dtok is None else _f32(dtok)
    dpool = None if dpool is None else _f32(dpool)
    dtable = torch.zeros((V, E), dtype=torch.float32, device=table.device)
    _cabi.call("cvcl_text_token_bwd", _p(ids), _p(lens), _p(table), _p(dtok), _p(dpool),
               float(pool_scale), _p(dtable), B, L, E, V, int(normalize), _stream())
    return dtable


@text_token_bwd.register_fake
def _(ids, lens, table, dtok, dpool, pool_scale, normalize):
    return table.new_empty(table.shape)


@torch.library.custom_op(_NS + "::embedding_gather", mutates_args=())
def embedding_gather(ids: Tensor, table: Tensor) -> Tensor:
    _need_cuda(ids, table)
    ids = _i64(ids); table = _f32(table)
    V, E = table.shape
    out = torch.empty(tuple(ids.shape) + (E,), dtype=torch.float32, device=table.device)
    _cabi.call("cvcl_embedding_gather", _p(ids), _p(table), _p(out), ids.numel(), E, V, _stream())
    return out


@embedding_gather.register_fake
def _(ids, table):
    return table.new_empty(tuple(ids.shape) + (table.shape[1],))


@torch.library.custom_op(_NS + "::embedding_scatter_add", mutates_args=())
def embedding_scatter_add(ids: Tensor, g: Tensor, V: int) -> Tensor:
    """autograd of embedding_gather: one gradient row per token."""
    _need_cuda(ids, g)
    ids = _i64(ids); g = _f32(g)
    E = g.shape[-1]
    n = ids.numel()
    dtable = torch.zeros((V, E), dtype=torch.float32, device=g.device)
    _cabi.call("cvcl_embedding_scatter_add", _p(ids), _p(g), _p(dtable), n, 1, E, V, 1, _stream())
    return dtable


@embedding_scatter_add.register_fake
def _(ids, g, V):
    return g.new_empty((V, g.shape[-1]))


class _TextFeaturesFlat(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ids, lens, table, normalize):
        feat, inv, _ = _raw(text_encoder_fwd)(ids, lens, table, normalize, False, 1.0)
        ctx.save_for_backward(ids, lens, feat, inv)
        ctx.normalize = normalize
        ctx.V = table.shape[0]
        return feat

    @staticmethod
    def backward(ctx, g):
        ids, lens, feat, inv = ctx.saved_tensors
        return None, None, _raw(embedding_bag_bwd)(ids, lens, g, feat, inv, ctx.normalize, ctx.V), None


class _TextFeaturesSpatial(torch.autograd.Function):
    """-> (tok [B,L,E] normalised per token, pooled [B,E] = sum_l tok * pool_scale / len)."""

    @staticmethod
    def forward(ctx, ids, lens, table, normalize, pool_scale, want_tok):
        pooled, inv, tok = _raw(text_encoder_fwd)(ids, lens, table, normalize, True, pool_scale, want_tok)
        ctx.save_for_backward(ids, lens, table)
        ctx.normalize = normalize
        ctx.pool_scale = pool_scale
        ctx.want_tok = want_tok
        if not want_tok:
            ctx.mark_non_differentiable(tok)
        return tok, pooled

    @staticmethod
    def backward(ctx, dtok, dpool):
        ids, lens, table = ctx.saved_tensors
        if not ctx.want_tok:
            dtok = None
        return None, None, _raw(text_token_bwd)(ids, lens, table, dtok, dpool, ctx.pool_scale,
                                          ctx.normalize), None, None, None


class _EmbeddingGather(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ids, table):
        ctx.save_for_backward(ids)
        ctx.V = table.shape[0]
        return _raw(embedding_gather)(ids, table)

    @staticmethod
    def backward(ctx, g):
        (ids,) = ctx.saved_tensors
        return None, _raw(embedding_scatter_add)(ids, g, ctx.V)


def text_features_flat(ids, lens, table, normalize=True):
    return _TextFeaturesFlat.apply(ids, lens, table, bool(normalize))


def text_features_spatial(ids, lens, table, normalize=True, pool_scale=1.0 / 49, want_tok=True):
    """-> (tok [B,L,E] | empty, pooled [B,E]); want_tok=False for the "mean" similarity (pooled only)."""
    return _TextFeaturesSpatial.apply(ids, lens, table, bool(normalize), float(pool_scale), bool(want_tok))


def text_outputs(ids, table):
    return _EmbeddingGather.apply(ids, table)


# ----------------------------------------------------------------------------------------
# K2 projection head
# ----------------------------------------------------------------------------------------
@torch.library.custom_op(_NS + "::head_proj_norm_fwd", mutates_args=())
def head_proj_norm_fwd(x: Tensor, w: Tensor, bias: Optional[Tensor], normalize: bool) -> Tuple[Tensor, Tensor]:
    """x [M,K] (fp32/bf16), w [E,K] -> (feat [M,E] fp32, inv_norm [M])."""
    _need_cuda(x, w)
    x16, _ = to_bf16_pair(x, False)
    w16, _ = to_bf16_pair(w, False)
    M, K = x16.shape
    E = w16.shape[0]
    b = None if bias is None else _f32(bias)
    feat = torch.empty((M, E), dtype=torch.float32, device=x.device)
    inv = torch.empty((M,), dtype=torch.float32, device=x.device)
    _cabi.call("cvcl_head_proj_norm_fwd", _p(x16), K, _p(w16), K, _p(b), M, E, K, int(normalize),
               _p(feat), E, None, 0, _p(inv), _stream())
    return feat, inv


@head_proj_norm_fwd.register_fake
def _(x, w, bias, normalize):
    return (x.new_empty((x.shape[0], w.shape[0]), dtype=torch.float32),
            x.new_empty((x.shape[0],), dtype=torch.float32))


@torch.library.custom_op(_NS + "::head_proj_norm_bwd", mutates_args=())
def head_proj_norm_bwd(g: Tensor, feat: Tensor, inv_norm: Tensor, x: Tensor, w: Tensor,
                       normalize: bool, need_dx: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (dW [E,K], db [E], dx [M,K] or empty), all fp32."""
    _need_cuda(g, x, w)
    g = _f32(g)
    M, E = g.shape
    K = x.shape[1]
    dev = g.device
    du16 = torch.empty((M, E), dtype=torch.bfloat16, device=dev)
    db = torch.zeros((E,), dtype=torch.float32, device=dev)
    _cabi.call("cvcl_rownorm_bwd", _p(g), _p(feat.contiguous()), _p(inv_norm), M, E, int(normalize),
               None, _p(du16), E, None, 0, _p(db), _stream())
    x16, _ = to_bf16_pair(x, False)
    dW = torch.empty((E, K), dtype=torch.float32, device=dev)
    _cabi.call("cvcl_head_weight_grad", _p(du16), E, _p(x16), K, E, K, M, _p(dW), K, _stream())
    if need_dx:
        w16, _ = to_bf16_pair(w, False)                     # [E,K] read MN-major: dx = du . W
        dx = torch.empty((M, K), dtype=torch.float32, device=dev)
        _cabi.call("cvcl_gemm_f32out", _p(du16), E, 0, _p(w16), K, 1, M, K, E, 1.0, _p(dx), K, _stream())
    else:
        dx = torch.empty((0,), dtype=torch.float32, device=dev)
    return dW, db, dx


@head_proj_norm_bwd.register_fake
def _(g, feat, inv_norm, x, w, normalize, need_dx):
    return (g.new_empty(w.shape, dtype=torch.float32), g.new_empty((w.shape[0],), dtype=torch.float32),
            g.new_empty(x.shape if need_dx else (0,), dtype=torch.float32))


def split_bf16_cat(x: Tensor, pattern: str) -> Tensor:
    """x [R, C] fp32 -> bf16 [R, 3C]: the two-term bf16 expansion x = hi + lo (hi = bf16(x), lo = bf16(x - hi))
    laid out along the contraction as `pattern` ("hlh" or "hhl").  With A as "hlh" and B as "hhl" one bf16 GEMM
    over 3C evaluates hi.hi + lo.hi + hi.lo with fp32 accumulation: the product to ~2^-16 relative instead of
    2^-8.  Used where a result feeds an ARG-MAX (spatial "max" similarity): near-tied candidates must be ordered
    as the reference's fp32 arithmetic orders them, or gradient rows move to other locations."""
    x = x.detach().float()
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    parts = {"h": hi, "l": lo}
    return torch.cat([parts[c] for c in pattern], dim=1).contiguous()


class _HeadFeatures(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, bias, normalize, split=False):
        if split and x.dtype == torch.float32:
            feat, inv = _raw(head_proj_norm_fwd)(split_bf16_cat(x, "hlh"), split_bf16_cat(w, "hhl"), bias, normalize)
        else:
            feat, inv = _raw(head_proj_norm_fwd)(x, w, bias, normalize)
        ctx.save_for_backward(x, w, feat, inv)
        ctx.normalize = normalize
        ctx.has_bias = bias is not None
        return feat

    @staticmethod
    def backward(ctx, g):
        x, w, feat, inv = ctx.saved_tensors
        need_dx = ctx.needs_input_grad[0]
        dW, db, dx = _raw(head_proj_norm_bwd)(g, feat, inv, x, w, ctx.normalize, need_dx)
        return (dx.to(x.dtype) if need_dx else None, dW.to(w.dtype),
                db if ctx.has_bias else None, None, None)


def head_features(x, w, bias, normalize=True, split=False):
    """normalise(x @ w.T + bias) on the tcgen05 engine; x [M,K] -> [M,E] fp32.  split=True: two-term bf16
    operands (see split_bf16_cat) -- fp32-grade features for consumers that take an arg-max."""
    return _HeadFeatures.apply(x, w, bias, bool(normalize), bool(split))


# ----------------------------------------------------------------------------------------
# spatial pooling (image factor of the "mean" similarity)
# ----------------------------------------------------------------------------------------
@torch.library.custom_op(_NS + "::spatial_pool", mutates_args=())
def spatial_pool_fwd(x: Tensor) -> Tensor:
    _need_cuda(x)
    x = _f32(x)
    B, HW, E = x.shape
    out = torch.empty((B, E), dtype=torch.float32, device=x.device)
    _cabi.call("cvcl_spatial_pool", _p(x), B, HW, E, _p(out), None, 0, None, 0, _stream())
    return out


@spatial_pool_fwd.register_fake
def _(x):
    return x.new_empty((x.shape[0], x.shape[2]))


class _SpatialPool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.hw = x.shape[1]
        return _raw(spatial_pool_fwd)(x)

    @staticmethod
    def backward(ctx, g):
        # the sum's gradient is a broadcast over the locations: materialised by one streaming-store kernel (returning
        # the expanded view instead made autograd copy it with a strided elementwise kernel: 62 us vs 17 at B = 1024)
        g = _f32(g)
        B, E = g.shape
        out = torch.empty((B, ctx.hw, E), dtype=torch.float32, device=g.device)
        _cabi.call("cvcl_spatial_pool_bwd", _p(g), B, ctx.hw, E, _p(out), _stream())
        return out


def spatial_pool(x):
    return _SpatialPool.apply(x)


def spatial_mean_factors(img_nhwc, ids, lens, table, normalize=True):
    """The two factors of the spatial "mean" similarity (multimodal.py:761-770: the mean over locations and words of
    <img[i,hw], tok[t,l]> factorises): (sum over the H*W locations of the image map [Bi,E], mean over the words of the
    normalised token rows / (H*W) [Bt,E]).  The text branch runs on a side stream beside the image branch (forward
    here; autograd replays each branch's backward on the stream its forward ran on), so under a CUDA graph the two
    become parallel branches."""
    HW = img_nhwc.shape[1]
    dev = img_nhwc.device
    main = torch.cuda.current_stream(dev)
    side = _side_stream(dev, 2)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        _, tpool = text_features_spatial(ids, lens, table, normalize, 1.0 / HW, want_tok=False)
    ipool = spatial_pool(img_nhwc)
    main.wait_stream(side)
    tpool.record_stream(main)
    return ipool, tpool


# ----------------------------------------------------------------------------------------
# K3 logits (materialised, for the forward() API)
# ----------------------------------------------------------------------------------------
@torch.library.custom_op(_NS + "::sim_logits_fwd", mutates_args=())
def sim_logits_fwd(img: Tensor, txt: Tensor, log_scale: float) -> Tuple[Tensor, Tensor]:
    _need_cuda(img, txt)
    i16, _ = to_bf16_pair(img, False)
    t16, _ = to_bf16_pair(txt, False)
    Ni, E = i16.shape
    Nt = t16.shape[0]
    lpi = torch.empty((Ni, Nt), dtype=torch.float32, device=img.device)
    lpt = torch.empty((Nt, Ni), dtype=torch.float32, device=img.device)
    _cabi.call("cvcl_sim_logits_fwd", _p(i16), _p(t16), E, Ni, Nt, E, float(log_scale), _p(lpi), _p(lpt),
               _stream())
    return lpi, lpt


@sim_logits_fwd.register_fake
def _(img, txt, log_scale):
    return (img.new_empty((img.shape[0], txt.shape[0]), dtype=torch.float32),
            img.new_empty((txt.shape[0], img.shape[0]), dtype=torch.float32))


@torch.library.custom_op(_NS + "::sim_logits_bwd", mutates_args=())
def sim_logits_bwd(g: Tensor, img: Tensor, txt: Tensor, log_scale: float) -> Tuple[Tensor, Tensor]:
    """g = d/d(lpi) + d/d(lpt)^T  [Ni,Nt] fp32 -> (dimg [Ni,E], dtxt [Nt,E]) fp32."""
    _need_cuda(g, img, txt)
    Ni, Nt = g.shape
    E = img.shape[1]
    ldg = _pad8(Nt)
    g32 = _f32(g)
    g16 = torch.empty((Ni, ldg), dtype=torch.bfloat16, device=g.device)
    _cabi.call("cvcl_cast_transpose", _p(g32), 0, _p(g16), None, 1, Ni, Nt, Nt, ldg, 0, 0, 0, 0, _stream())
    i16, _ = to_bf16_pair(img, False)
    t16, _ = to_bf16_pair(txt, False)
    scale = math.exp(log_scale)
    dimg = torch.empty((Ni, E), dtype=torch.float32, device=g.device)
    dtxt = torch.empty((Nt, E), dtype=torch.float32, device=g.device)
    # dimg = g . txt (txt read MN-major);  dtxt = g^T . img (g and img both read MN-major)
    _cabi.call("cvcl_gemm_f32out", _p(g16), ldg, 0, _p(t16), E, 1, Ni, E, Nt, scale, _p(dimg), E, _stream())
    _cabi.call("cvcl_gemm_f32out", _p(g16), ldg, 1, _p(i16), E, 1, Nt, E, Ni, scale, _p(dtxt), E, _stream())
    return dimg, dtxt


@sim_logits_bwd.register_fake
def _(g, img, txt, log_scale):
    return (img.new_empty(img.shape, dtype=torch.float32), txt.new_empty(txt.shape, dtype=torch.float32))


class _SimLogits(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img, txt, s):
        ls = _scalar(s)
        lpi, lpt = _raw(sim_logits_fwd)(img, txt, ls)
        ctx.save_for_backward(img, txt, lpi)
        ctx.ls = ls
        ctx.s_is_tensor = torch.is_tensor(s)
        return lpi, lpt

    @staticmethod
    def backward(ctx, glpi, glpt):
        img, txt, lpi = ctx.saved_tensors
        g = glpi + glpt.t()
        dimg, dtxt = _raw(sim_logits_bwd)(g, img, txt, ctx.ls)
        ds = (g * lpi).sum() if ctx.s_is_tensor and ctx.needs_input_grad[2] else None
        return dimg.to(img.dtype), dtxt.to(txt.dtype), ds


def sim_logits(img, txt, s):
    """(logits_per_image [Ni,Nt], logits_per_text [Nt,Ni]) = exp(s) * img @ txt.T (+ transpose)."""
    return _SimLogits.apply(img, txt, s)


# ----------------------------------------------------------------------------------------
# K3+K4+K5: fused similarity + symmetric InfoNCE at feature level (single GPU or one shard)
# ----------------------------------------------------------------------------------------
@torch.library.custom_op(_NS + "::sim_infonce_fwd", mutates_args=())
def sim_infonce_fwd(img_q: Tensor, txt_k: Tensor, txt_q: Tensor, img_k: Tensor, log_scale: float,
                    diag_off: int, inv_rows: float, unit_norm: bool = False
                    ) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """bf16 operands [.,E] -> (out5 [8] fp32, lse0 [M0], lse1 [M1], argmax0 [M0], argmax1 [M1]).
    unit_norm: the rows are unit vectors (F.normalize) -- large single-device problems then take one similarity
    pass for both directions (see cvcl_sim_infonce_fwd)."""
    _need_cuda(img_q, txt_k, txt_q, img_k)
    M0, E = img_q.shape
    N0 = txt_k.shape[0]
    M1 = txt_q.shape[0]
    N1 = img_k.shape[0]
    dev = img_q.device
    lib = _cabi.load()
    ws = torch.empty((lib.cvcl_sim_workspace_bytes(M0, N0, M1, N1),), dtype=torch.uint8, device=dev)
    out5 = torch.zeros((8,), dtype=torch.float32, device=dev)
    lse0 = torch.empty((M0,), dtype=torch.float32, device=dev)
    lse1 = torch.empty((M1,), dtype=torch.float32, device=dev)
    a0 = torch.empty((M0,), dtype=torch.int32, device=dev)
    a1 = torch.empty((M1,), dtype=torch.int32, device=dev)
    _cabi.call("cvcl_sim_infonce_fwd", _p(img_q), _p(txt_k), _p(txt_q), _p(img_k), E, M0, N0, M1, N1, E,
               float(log_scale), int(diag_off), float(inv_rows), _p(ws), _p(lse0), _p(lse1), _p(a0), _p(a1),
               _p(out5), int(bool(unit_norm)), _stream())
    return out5, lse0, lse1, a0, a1


@sim_infonce_fwd.register_fake
def _(img_q, txt_k, txt_q, img_k, log_scale, diag_off, inv_rows, unit_norm=False):
    f = dict(dtype=torch.float32)
    return (img_q.new_empty((8,), **f), img_q.new_empty((img_q.shape[0],), **f),
            img_q.new_empty((txt_q.shape[0],), **f),
            img_q.new_empty((img_q.shape[0],), dtype=torch.int32),
            img_q.new_empty((txt_q.shape[0],), dtype=torch.int32))


@torch.library.custom_op(_NS + "::sim_infonce_bwd", mutates_args=())
def sim_infonce_bwd(img_q: Tensor, txt_k: Tensor, txt_q: Tensor, img_k: Tensor, log_scale: float,
                    diag_off: int, coef: float, lse_q0: Tensor, lse_k0: Tensor, lse_q1: Tensor,
                    lse_k1: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (dimg_q [M0,E] fp32, dtxt_q [M1,E] fp32, dscale [1] fp32 (local rows only))."""
    _need_cuda(img_q, txt_k, txt_q, img_k)
    M0, E = img_q.shape
    N0 = txt_k.shape[0]
    M1 = txt_q.shape[0]
    N1 = img_k.shape[0]
    dev = img_q.device
    # one GPU: queries and keys are the same tensors.  (A shard whose local block sits at offset 0 of the gathered
    # buffer shares the POINTER with it -- rank 0 -- so the shapes must agree too.)
    single = (img_q.data_ptr() == img_k.data_ptr() and txt_q.data_ptr() == txt_k.data_ptr()
              and M0 == N1 and M1 == N0)
    ld0, ld1 = _pad8(N0), _pad8(N1)
    G0 = torch.empty((M0, ld0), dtype=torch.bfloat16, device=dev)
    G1 = None if single else torch.empty((M1, ld1), dtype=torch.bfloat16, device=dev)
    ds = torch.zeros((1,), dtype=torch.float32, device=dev)
    # the diagonal of G in fp32, per row: G_ii - bf16(Gs_ii) (dT of one GPU reads Gs0^T, whose diagonal is gd0's)
    gd0 = torch.empty((M0,), dtype=torch.float32, device=dev)
    gd1 = gd0 if single else torch.empty((M1,), dtype=torch.float32, device=dev)
    _cabi.call("cvcl_sim_infonce_bwd_g", _p(img_q), _p(txt_k), _p(txt_q), _p(img_k), E, M0, N0, M1, N1, E,
               float(log_scale), int(diag_off), float(coef), _p(lse_q0), _p(lse_k0), _p(lse_q1), _p(lse_k1),
               _p(G0), ld0, _p(G1), ld1, _p(gd0), None if single else _p(gd1), _p(ds), _stream())
    dimg = torch.empty((M0, E), dtype=torch.float32, device=dev)
    dtxt = torch.empty((M1, E), dtype=torch.float32, device=dev)
    if min(N0, N1) >= 4096:
        # long contraction: plain 128 x 256-tile GEMMs (higher tensor throughput), then the fp32
        # diagonal term as one addcmul over [M,E]
        _cabi.call("cvcl_gemm_f32out", _p(G0), ld0, 0, _p(txt_k), E, 1, M0, E, N0, 1.0, _p(dimg), E, _stream())
        if single:
            _cabi.call("cvcl_gemm_f32out", _p(G0), ld0, 1, _p(img_k), E, 1, M1, E, N1, 1.0, _p(dtxt), E, _stream())
        else:
            _cabi.call("cvcl_gemm_f32out", _p(G1), ld1, 0, _p(img_k), E, 1, M1, E, N1, 1.0, _p(dtxt), E, _stream())
        dimg.addcmul_(txt_k[diag_off:diag_off + M0].float(), gd0[:, None])
        dtxt.addcmul_(img_k[diag_off:diag_off + M1].float(), gd1[:, None])
        return dimg, dtxt, ds
    _cabi.call("cvcl_feat_grad_norm_bwd", _p(G0), ld0, 0, _p(txt_k), E, M0, E, N0, None, 0, None, 0, None,
               _p(txt_k), E, N0, int(diag_off), _p(gd0), _p(dimg), E, None, 0, None, _stream())
    if single:      # dT = Gs^T . I: the same Gs read MN-major, no second orientation needed
        _cabi.call("cvcl_feat_grad_norm_bwd", _p(G0), ld0, 1, _p(img_k), E, M1, E, N1, None, 0, None, 0, None,
                   _p(img_k), E, N1, int(diag_off), _p(gd1), _p(dtxt), E, None, 0, None, _stream())
    else:
        _cabi.call("cvcl_feat_grad_norm_bwd", _p(G1), ld1, 0, _p(img_k), E, M1, E, N1, None, 0, None, 0, None,
                   _p(img_k), E, N1, int(diag_off), _p(gd1), _p(dtxt), E, None, 0, None, _stream())
    return dimg, dtxt, ds


@sim_infonce_bwd.register_fake
def _(img_q, txt_k, txt_q, img_k, log_scale, diag_off, coef, lse_q0, lse_k0, lse_q1, lse_k1):
    f = dict(dtype=torch.float32)
    return (img_q.new_empty(img_q.shape, **f), txt_q.new_empty(txt_q.shape, **f), img_q.new_empty((1,), **f))


class _SimInfoNCE(torch.autograd.Function):
    """Symmetric InfoNCE on (local) features; with a process group the features are all-gathered
    and each rank evaluates its row block and column block (sharding.py, SURVEY section 8e).
    Returns the five GLOBAL scalars (identical on all ranks).  Gradients: d img / d txt for the
    local pairs are complete; d s is summed over ranks so every rank holds the full value."""

    @staticmethod
    def forward(ctx, img, txt, s, group, unit_norm=False):
        from . import sharding
        i16, _ = to_bf16_pair(img, False)
        t16, _ = to_bf16_pair(txt, False)
        fwd = _raw(sim_infonce_fwd)
        if unit_norm:
            def fwd(*a, _f=_raw(sim_infonce_fwd)):
                return _f(*a, True)
        out5, saved, (a0, a1) = sharding.infonce_forward(i16, t16, _scalar(s), group, fwd)
        ctx.saved = saved
        ctx.group = group
        ctx.meta = (img.dtype, txt.dtype, torch.is_tensor(s))
        ctx.set_materialize_grads(False)          # only the loss is differentiated: no zero gradients for the metrics
        o = out5[:5].unbind(0)
        ctx.mark_non_differentiable(o[1], o[2], o[3], o[4], a0, a1)
        return o[0], o[1], o[2], o[3], o[4], a0, a1

    @staticmethod
    def backward(ctx, gloss, *unused):
        from . import sharding
        if gloss is None:
            return None, None, None, None, None
        idt, tdt, s_is_tensor = ctx.meta
        dimg, dtxt, ds = sharding.infonce_backward(ctx.saved, ctx.group, _raw(sim_infonce_bwd))
        dimg = (dimg * gloss).to(idt)
        dtxt = (dtxt * gloss).to(tdt)
        ds_out = (ds[0] * gloss) if (s_is_tensor and ctx.needs_input_grad[2]) else None
        return dimg, dtxt, ds_out, None, None


def sim_infonce(img, txt, s, group=None, unit_norm=False):
    """-> (loss, image_accuracy, text_accuracy, image_entropy, text_entropy, image_pred, text_pred).
    unit_norm=True: img / txt rows are unit vectors (the output of F.normalize); lets large single-device batches
    evaluate the similarity once for both directions."""
    return _SimInfoNCE.apply(img, txt, s, group, bool(unit_norm))


# ----------------------------------------------------------------------------------------
# fused flat train step (K1..K5 sequenced inside one C call)
# ----------------------------------------------------------------------------------------
def split_flat_grads(flat: Tensor, E: int, K: int, V: int):
    """views into the flat gradient buffer [ds(4) | db(E) | dtable(V*E) | dW(E*K)] (one split op + three views)."""
    n = 4 + E + V * E + E * K
    if flat.numel() != n:
        flat = flat[:n]
    ds4, db, dt, dw = flat.split_with_sizes((4, E, V * E, E * K))
    return ds4[0:1], db, dt.view(V, E), dw.view(E, K)


# bf16 shadows of fp32 master weights, keyed by storage: recast only when the parameter's version changed
# (an optimizer step).  `register_weight_shadow` lets an optimizer that writes the shadow itself
# (FusedAdamW: cvcl_adamw_step's bf16_shadow output) hand it over, so no cast runs at all.
_SHADOWS = {}
_FUSED_WS = {}
FUSED_STEP = True          # False: always use the multi-kernel step, single-GPU and sharded


def _shadow_entry(w):
    ent = _SHADOWS.get(id(w))
    if ent is not None and (ent[0]() is not w or ent[1] != w.data_ptr()):
        ent = None                                   # id reused by another tensor / storage swapped
    return ent


def register_weight_shadow(w: Tensor, w16: Tensor):
    """w16 (bf16, same shape) is kept equal to bf16(w) by its owner from now on (e.g. FusedAdamW, whose
    kernel writes the refreshed shadow together with the fp32 master)."""
    import weakref
    key = id(w)
    _SHADOWS[key] = [weakref.ref(w, lambda _r, k=key: _SHADOWS.pop(k, None)), w.data_ptr(), None, w16]


def drop_weight_shadow(w: Tensor):
    _SHADOWS.pop(id(w), None)


def weight_shadow(w: Tensor) -> Tensor:
    """bf16 copy of the fp32 master weight `w` [E,K]: one cast per parameter version (an optimizer step
    bumps the version), none at all when an owner registered the shadow."""
    import weakref
    ent = _shadow_entry(w)
    ver = w._version
    if ent is not None and (ent[2] is None or ent[2] == ver):
        return ent[3]
    w32 = _f32(w)
    if torch.cuda.is_current_stream_capturing():
        # a capture must not bake in "no cast needed": cast inside the graph into a private buffer
        return to_bf16_pair(w32, False)[0]
    w16 = ent[3] if ent is not None else torch.empty(w.shape, dtype=torch.bfloat16, device=w.device)
    R, C = w.shape
    _cabi.call("cvcl_cast_transpose", _p(w32), 0, _p(w16), None, 1, R, C, C, C, 0, 0, 0, 0, _stream())
    key = id(w)
    _SHADOWS[key] = [weakref.ref(w, lambda _r, k=key: _SHADOWS.pop(k, None)), w.data_ptr(), ver, w16]
    return w16


def _fused_workspace(dev, B, L, E, K, V):
    """persistent, zero-initialised workspace of the one-kernel step (one step in flight per device and
    shape; calls on one stream are ordered, which is how a training loop uses it)."""
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), B, L, E, K, V)
    ws = _FUSED_WS.get(key)
    if ws is None:
        nbytes = int(_cabi.load().cvcl_flat_fused_workspace_bytes(B, L, E, K, V))
        ws = _FUSED_WS[key] = torch.zeros((nbytes,), dtype=torch.uint8, device=dev)
    return ws


_FUSED_OK = {}


def fused_supported(B, L, E, K, V) -> bool:
    if not FUSED_STEP:
        return False
    key = (B, L, E, K, V)
    ok = _FUSED_OK.get(key)
    if ok is None:
        ok = _FUSED_OK[key] = bool(_cabi.load().cvcl_flat_fused_supported(B, L, E, K, V))
    return ok


def flat_step_layout(B, L, E, K, V):
    """workspace block offsets of the multi-kernel step after it ran (see cvcl_flat_step_layout)."""
    import ctypes
    arr = (ctypes.c_longlong * 12)()
    _cabi.call("cvcl_flat_step_layout", B, L, E, K, V, arr, 12)
    names = ["img16", "txt16", "invn_i", "invn_t", "lse0", "lse1", "G0", "du16", "dm", "gdiag", "ldB", "bytes"]
    return dict(zip(names, [int(v) for v in arr]))


def fused_layout(B, L, E, K, V):
    """workspace block offsets of the one-kernel step (see cvcl_flat_fused_layout)."""
    import ctypes
    arr = (ctypes.c_longlong * 25)()
    _cabi.call("cvcl_flat_fused_layout", B, L, E, K, V, arr, 25)
    names = ["ctrl", "hpart", "img16", "txt16", "invn", "part", "diag", "lse", "rb_part", "dspart", "dqpart",
             "du16", "dbpart", "bytes", "Bp", "KS", "nPart", "dw_bn", "grid", "nCB", "dm16", "cmat", "QS", "Vp",
             "gdiag"]
    return dict(zip(names, [int(v) for v in arr]))


@torch.library.custom_op(_NS + "::flat_contrastive_step", mutates_args=())
def flat_contrastive_step(x: Tensor, ids: Tensor, lens: Tensor, w: Tensor, bias: Tensor, table: Tensor,
                          log_scale: float, normalize: bool, need_grads: bool, want_features: bool,
                          log_scale_t: Optional[Tensor] = None, phase_limit: int = 0
                          ) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """-> (out5 [8], img_feat [B,E] | empty, txt_feat [B,E] | empty, grads_flat | empty); the flat
    buffer holds [ds(4) | db(E) | dtable(V*E) | dW(E*K)] (see split_flat_grads): one all-reduce when
    sharded.  log_scale_t: optional CUDA scalar s read on the device (no host sync; one-kernel path).
    Shapes the persistent kernel covers (cvcl_flat_fused_supported) run as ONE launch; others as the
    multi-kernel sequence of cvcl_flat_contrastive_step."""
    _need_cuda(x, ids, lens, w, bias, table)
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    x = x.detach().contiguous()
    ids = _i64(ids); lens = _i64(lens)
    w_param = w
    w = _f32(w); bias = _f32(bias); table = _f32(table)
    B, K = x.shape
    L = ids.shape[1]
    V, E = table.shape
    dev = x.device
    lib = _cabi.load()
    f32 = dict(dtype=torch.float32, device=dev)
    out5 = torch.empty((8,), **f32)
    img_f = torch.empty((B, E), **f32) if want_features else torch.empty((0,), **f32)
    txt_f = torch.empty((B, E), **f32) if want_features else torch.empty((0,), **f32)
    if need_grads:
        flat = torch.empty((4 + E + V * E + E * K,), **f32)
    else:
        flat = torch.empty((0,), **f32)
    if fused_supported(B, L, E, K, V):
        x16, _ = to_bf16_pair(x, False)
        w16 = weight_shadow(w_param)
        ws = _fused_workspace(dev, B, L, E, K, V)
        # gradient pointers straight from the layout of the flat buffer (split_flat_grads): no views on this path
        g0 = flat.data_ptr() if need_grads else None
        _cabi.call("cvcl_flat_step_fused", _p(x16), _p(w16), _p(ids), _p(lens), _p(bias), _p(table),
                   B, L, E, K, V, int(normalize), float(log_scale), _p(log_scale_t), int(need_grads),
                   _p(ws), _p(out5), _p(img_f) if want_features else None,
                   _p(txt_f) if want_features else None,
                   g0 + 4 * (4 + E + V * E) if need_grads else None, g0 + 16 if need_grads else None,
                   g0 + 4 * (4 + E) if need_grads else None, g0, _p(token_status(dev)), int(phase_limit), _stream())
        return out5, img_f, txt_f, flat
    if need_grads:
        ds, db, dtable, dW = split_flat_grads(flat, E, K, V)
    else:
        ds = db = dtable = dW = None
    if log_scale_t is not None:
        log_scale = float(log_scale_t)               # multi-kernel path: host scalar (one D2H sync)
    out5.zero_()
    ws = torch.empty((lib.cvcl_flat_step_workspace_bytes(B, L, E, K, V),), dtype=torch.uint8, device=dev)
    _cabi.call("cvcl_flat_contrastive_step", _p(x), int(x.dtype == torch.bfloat16), _p(ids), _p(lens),
               _p(w), _p(bias), _p(table), B, L, E, K, V, int(normalize), float(log_scale),
               int(need_grads), _p(ws), _p(out5), _p(img_f) if want_features else None,
               _p(txt_f) if want_features else None, _p(dW), _p(db), _p(dtable), _p(ds), None, _stream())
    return out5, img_f, txt_f, flat


@flat_contrastive_step.register_fake
def _(x, ids, lens, w, bias, table, log_scale, normalize, need_grads, want_features, log_scale_t=None,
      phase_limit=0):
    f = dict(dtype=torch.float32)
    B, K = x.shape
    V, E = table.shape

    def feat():
        return x.new_empty((B, E) if want_features else (0,), **f)
    return (x.new_empty((8,), **f), feat(), feat(),
            x.new_empty((4 + E + V * E + E * K) if need_grads else 0, **f))


class _FlatContrastiveStep(torch.autograd.Function):
    """loss and all parameter gradients in one pass; backward only scales the saved gradients by
    the upstream scalar (the loss is a scalar, so d(c*loss)/dtheta = c * dloss/dtheta)."""

    @staticmethod
    def forward(ctx, x, ids, lens, w, bias, table, s, normalize, want_features):
        need = any(t is not None and torch.is_tensor(t) and t.requires_grad for t in (w, bias, table, s))
        if torch.is_tensor(x) and x.requires_grad:
            raise RuntimeError("flat_contrastive_step does not produce d/dx; use the op-by-op path "
                               "(finetune_cnn=True) instead")
        # a CUDA scalar s (trainable temperature) is read on the device: no .item() sync per step
        s_dev = s.detach().reshape(1).float() if (torch.is_tensor(s) and s.is_cuda) else None
        out5, img_f, txt_f, flat = _raw(flat_contrastive_step)(
            x, ids, lens, w, bias, table, 0.0 if s_dev is not None else _scalar(s), normalize, need,
            want_features, s_dev)
        ctx.need = need
        ctx.consumed = False
        ctx.s_is_tensor = torch.is_tensor(s)
        ctx.dims = (table.shape[1], x.shape[1], table.shape[0])
        if need:
            ctx.save_for_backward(flat)
        # only the loss carries a gradient: the other scalars are metrics.  Without this the engine materialises a
        # zero gradient for each unused output on every backward (four fill kernels per step in the launch list)
        ctx.set_materialize_grads(False)
        o = out5.unbind(0)                       # one op for the five scalars
        ctx.mark_non_differentiable(o[1], o[2], o[3], o[4], img_f, txt_f)
        return o[0], o[1], o[2], o[3], o[4], img_f, txt_f

    @staticmethod
    def backward(ctx, gloss, *unused):
        if not ctx.need or gloss is None:
            return (None,) * 9
        (flat,) = ctx.saved_tensors
        E, K, V = ctx.dims
        # the gradients were computed for upstream = 1; scale in place (no 9.6 MB temporary).  Marked so a
        # second backward through the same graph (retain_graph) is rejected instead of scaling twice.
        if ctx.consumed:
            raise RuntimeError("flat_contrastive_step: backward through this step a second time is not supported")
        ctx.consumed = True
        flat.mul_(gloss)
        ds, db, dtable, dW = split_flat_grads(flat, E, K, V)
        return (None, None, None, dW, db, dtable, ds[0] if ctx.s_is_tensor else None, None, None)


def flat_contrastive_loss(x, ids, lens, w, bias, table, s, normalize=True, want_features=False, group=None):
    """-> (loss, img_acc, txt_acc, img_ent, txt_ent, img_feat|empty, txt_feat|empty).
    group: torch.distributed process group -> global-batch InfoNCE over the ranks (the returned
    scalars are global; parameter gradients are already summed over ranks)."""
    if group is not None:
        return _FlatContrastiveStepSharded.apply(x, ids, lens, w, bias, table, s, bool(normalize),
                                                 bool(want_features), group)
    return _FlatContrastiveStep.apply(x, ids, lens, w, bias, table, s, bool(normalize),
                                      bool(want_features))


def flat_step_sharded(x, ids, lens, w, bias, table, log_scale, normalize, need_grads, want_features, group,
                      stats_slot=0):
    """The flat train step with the batch sharded by pairs over `group` (SURVEY 8e): local encoders,
    ONE all-gather of the bf16 [img|txt] features, row-block + column-block InfoNCE, one all-gather of
    the LSEs, local backward, ONE all-reduce of [out5 | ds | db | dtable | dW].
    -> (stats_flat, img_feat | None, txt_feat | None); stats_flat = [out5(8) | split_flat_grads layout].
    With the peer-memory exchange (sharding.PeerExchange) the three collectives are single kernels over
    NVLink peer memory and stats_flat is the persistent symmetric block `stats_slot`: valid until the
    next call with the same slot."""
    from . import sharding
    _need_cuda(x, ids, lens, w, bias, table)
    world, rank = sharding.group_info(group)
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    x = x.detach().contiguous()
    ids = _i64(ids); lens = _i64(lens)
    w_param = w
    w = _f32(w); bias = _f32(bias); table = _f32(table)
    B, K = x.shape
    L = ids.shape[1]
    V, E = table.shape
    Bg = B * world
    dev = x.device
    lib = _cabi.load()
    C = _cabi.call
    st = _stream()
    bf = dict(dtype=torch.bfloat16, device=dev); f32 = dict(dtype=torch.float32, device=dev)
    main = torch.cuda.current_stream(dev)
    side = _side_stream(dev)
    n_g = 4 + E + V * E + E * K
    n_stats = 8 + (n_g if need_grads else 0)
    # the three collectives run over peer-mapped symmetric memory when available (sharding.PeerExchange):
    # the arena is sized for the training step and shared with the forward-only call
    use_fused = world > 1 and FUSED_STEP and bool(lib.cvcl_flat_fused_sharded_supported(B, L, E, K, V, world))
    # (the one-kernel step keeps its per-tile gradient scratch in the same arena)
    min_scr = int(lib.cvcl_flat_fused_sharded_scratch_bytes(B, L, E, K, V, world)) if use_fused else 0
    px = sharding.PeerExchange.get(group, B, E, 8 + n_g, dev, min_scr) if world > 1 else None
    if px is not None and use_fused:
        # ---- ONE persistent kernel per rank: the producing phases store features / LSEs into every rank's gathered
        # buffers over NVLink, its grid barriers span the ranks, and its last phase sums the gradients over the ranks
        x16, _ = to_bf16_pair(x, False)
        w16 = weight_shadow(w_param)
        key = ("sharded", dev.index if dev.index is not None else torch.cuda.current_device(), B, L, E, K, V, world)
        ws = _FUSED_WS.get(key)
        if ws is None:
            ws = _FUSED_WS[key] = torch.zeros((int(lib.cvcl_flat_fused_sharded_workspace_bytes(B, L, E, K, V, world)),),
                                              dtype=torch.uint8, device=dev)
        stats = px.stats[stats_slot][:8 + n_g]
        img_f = torch.empty((B, E), **f32) if want_features else None
        txt_f = torch.empty((B, E), **f32) if want_features else None
        ds, db, dtable, dW = split_flat_grads(stats[8:], E, K, V)
        C("cvcl_flat_step_fused_sharded", _p(x16), _p(w16), _p(ids), _p(lens), _p(bias), _p(table), B, L, E, K, V,
          int(normalize), float(log_scale), None, int(need_grads), _p(ws), _p(stats), _p(img_f), _p(txt_f),
          _p(dW) if need_grads else None, _p(db) if need_grads else None, _p(dtable) if need_grads else None,
          _p(ds) if need_grads else None, _p(token_status(dev)), 0, world, rank, px.p_txt_all, px.p_img_all, px.p_part_all,
          px.p_flags[px.CH_FUSED], px.fused_epoch.data_ptr(),
          # the kernel's last phase sums [out5 | ds | db | d table | dW] over the ranks in place (two-shot, push, fixed
          # rank order) and its closing cross-rank barrier lets the next step overwrite the exchange buffers; a
          # forward-only step sums just the five scalars
          px.p_stats[stats_slot], px.p_scratch, n_stats if need_grads else 8, st)
        return stats[:n_stats], img_f, txt_f
    # [img | txt] per pair: one exchange moves both
    feats = px.feats if px is not None else torch.empty((B, 2 * E), **bf)
    img_l, txt_l = feats[:, :E], feats[:, E:]
    invn_i = torch.empty((B,), **f32); invn_t = torch.empty((B,), **f32)
    img_f = torch.empty((B, E), **f32) if want_features else None
    txt_f = torch.empty((B, E), **f32) if want_features else None
    # with the peer exchange `stats` is the persistent symmetric block: valid until the next call
    stats = px.stats[stats_slot][:n_stats] if px is not None else torch.empty((n_stats,), **f32)
    # ---- forward: text encoder + accumulator zeroing (side) || cast W -> head GEMM (main)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        C("cvcl_text_encoder_fwd", _p(ids), _p(lens), _p(table), B, L, E, V, int(normalize), 0, 1.0,
          _p(txt_f), _p(txt_l), 2 * E, _p(invn_t), None, None, None, side.cuda_stream)
    zero = _side_stream(dev, 1)          # third branch: the 9.6 MB accumulator memset is off both critical paths
    zero.wait_stream(main)
    with torch.cuda.stream(zero):
        stats.zero_()
    w16 = torch.empty((E, K), **bf)
    C("cvcl_cast_transpose", _p(w), 0, _p(w16), None, 1, E, K, K, K, 0, 0, 0, 0, st)
    x16, _ = to_bf16_pair(x, False)
    img_u = img_f if img_f is not None else torch.empty((B, E), **f32)   # fp32 out = split-K accumulator
    C("cvcl_head_proj_norm_fwd", _p(x16), K, _p(w16), K, _p(bias), B, E, K, int(normalize), _p(img_u), E,
      _p(img_l), 2 * E, _p(invn_i), st)
    main.wait_stream(side)
    if px is not None:       # one kernel: 16-byte stores into every rank's gathered buffer (NVLink) + barrier
        feats_all = px.gather_feats(st)
    else:
        feats_all = sharding.all_gather_rows(feats, group, world)      # [Bg, 2E] (NCCL)
    img_a, txt_a = feats_all[:, :E], feats_all[:, E:]
    main.wait_stream(zero)               # the similarity kernel accumulates out5 into stats[0:8]
    ws = torch.empty((lib.cvcl_sim_workspace_bytes(B, Bg, B, Bg),), dtype=torch.uint8, device=dev)
    lse = px.lse if px is not None else torch.empty((2, B), **f32)
    C("cvcl_sim_infonce_fwd", _p(img_l), _p(txt_a), _p(txt_l), _p(img_a), 2 * E, B, Bg, B, Bg, E,
      float(log_scale), rank * B, 1.0 / Bg, _p(ws), _p(lse[0]), _p(lse[1]), None, None, _p(stats), 0, st)
    if need_grads:
        if px is not None:
            lse_all = px.gather_lse(st)
        elif world > 1:
            lse_all = sharding.all_gather_rows(lse, group, world).view(world, 2, B).permute(1, 0, 2).contiguous()
        else:
            lse_all = lse
        lse0_all, lse1_all = lse_all[0].reshape(-1), lse_all[1].reshape(-1)
        ds, db, dtable, dW = split_flat_grads(stats[8:], E, K, V)
        ldg = _pad8(Bg)
        G0 = torch.empty((B, ldg), **bf); G1 = torch.empty((B, ldg), **bf)
        gdiag = torch.empty((2, B), **f32)          # per row: G_ii - bf16(Gs_ii) of each direction
        coef = 0.5 / Bg
        C("cvcl_sim_infonce_bwd_g", _p(img_l), _p(txt_a), _p(txt_l), _p(img_a), 2 * E, B, Bg, B, Bg, E,
          float(log_scale), rank * B, coef, _p(lse[0]), _p(lse1_all), _p(lse[1]), _p(lse0_all),
          _p(G0), ldg, _p(G1), ldg, _p(gdiag[0]), _p(gdiag[1]), _p(ds), st)
        du16 = torch.empty((B, E), **bf); dm = torch.empty((B, E), **f32)
        # ---- backward: dT -> embedding scatter (side) || dI -> dW (main)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            ss = side.cuda_stream
            C("cvcl_feat_grad_norm_bwd", _p(G1), ldg, 0, _p(img_a), 2 * E, B, E, Bg, _p(txt_l), 2 * E, _p(invn_t),
              int(normalize), _p(lens), _p(img_a), 2 * E, Bg, rank * B, _p(gdiag[1]), _p(dm), E, None, 0, None, ss)
            C("cvcl_embedding_scatter_add", _p(ids), _p(dm), _p(dtable), B, L, E, V, 0, ss)
        # long contraction (Bg >= 1536): the library splits it over the SMs into this fp32 scratch
        acc_i = torch.empty((B, E), **f32) if Bg >= 1536 else None
        C("cvcl_feat_grad_norm_bwd_ws", _p(G0), ldg, 0, _p(txt_a), 2 * E, B, E, Bg, _p(img_l), 2 * E, _p(invn_i),
          int(normalize), None, _p(txt_a), 2 * E, Bg, rank * B, _p(gdiag[0]), None, 0, _p(du16), E, _p(db), _p(acc_i), st)
        C("cvcl_head_weight_grad", _p(du16), E, _p(x16), K, E, K, B, _p(dW), K, st)
        main.wait_stream(side)        # every side-stream use is ordered before anything that follows
    if px is not None:       # one kernel: barrier, two-shot in-place sum over peer memory, barrier
        px.allreduce_stats(stats_slot, n_stats, st)
    elif world > 1:
        import torch.distributed as dist
        dist.all_reduce(stats, group=group)
    return stats, img_f, txt_f


_SIDE_STREAMS = {}


def _side_stream(dev, which=0):
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device(), which)
    s = _SIDE_STREAMS.get(key)
    if s is None:
        s = _SIDE_STREAMS[key] = torch.cuda.Stream(device=dev)
    return s


class _FlatContrastiveStepSharded(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ids, lens, w, bias, table, s, normalize, want_features, group):
        need = any(t is not None and torch.is_tensor(t) and t.requires_grad for t in (w, bias, table, s))
        if torch.is_tensor(x) and x.requires_grad:
            raise RuntimeError("the sharded flat step does not produce d/dx; use train_path='ops'")
        stats, img_f, txt_f = flat_step_sharded(x, ids, lens, w, bias, table, _scalar(s), normalize, need,
                                                want_features, group)
        if stats._base is not None:       # persistent symmetric block (peer exchange): the caller owns a copy
            stats = stats.clone()
        ctx.need = need
        ctx.s_is_tensor = torch.is_tensor(s)
        ctx.dims = (table.shape[1], x.shape[1], table.shape[0])
        if need:
            ctx.save_for_backward(stats)
        e = stats.new_empty((0,))
        img_f = e if img_f is None else img_f
        txt_f = e.clone() if txt_f is None else txt_f
        ctx.set_materialize_grads(False)
        o = stats[:5].unbind(0)
        ctx.mark_non_differentiable(o[1], o[2], o[3], o[4], img_f, txt_f)
        return o[0], o[1], o[2], o[3], o[4], img_f, txt_f

    @staticmethod
    def backward(ctx, gloss, *unused):
        if not ctx.need or gloss is None:
            return (None,) * 10
        (stats,) = ctx.saved_tensors
        E, K, V = ctx.dims
        ds, db, dtable, dW = split_flat_grads(stats[8:] * gloss, E, K, V)
        return (None, None, None, dW, db, dtable, ds[0] if ctx.s_is_tensor else None, None, None, None)


def linear_f32(x: Tensor, w: Tensor, bias: Optional[Tensor]) -> Tensor:
    """x [M,K] . w[N,K]^T + bias in fp32 with fp32 accumulation (cvcl_linear_f32): the exact-mode projection head
    of the evaluation path (no tensor cores, no library GEMM)."""
    if x.dim() != 2 or w.dim() != 2 or w.shape[1] != x.shape[1]:
        raise ValueError("linear_f32: x %s and w %s do not fit (need x [M,K], w [N,K])"
                         % (tuple(x.shape), tuple(w.shape)))
    if bias is not None and tuple(bias.shape) != (w.shape[0],):
        raise ValueError("linear_f32: bias %s does not fit w %s" % (tuple(bias.shape), tuple(w.shape)))
    _need_cuda(x, w, bias)
    x = _f32(x); w = _f32(w)
    bias = _f32(bias) if bias is not None else None
    M, K = x.shape
    N = w.shape[0]
    out = torch.empty((M, N), dtype=torch.float32, device=x.device)
    _cabi.call("cvcl_linear_f32", _p(x), K, _p(w), K, _p(bias), M, N, K, _p(out), N, _stream())
    return out


def normalize_rows_f32(x: Tensor) -> Tensor:
    """F.normalize(x, dim=-1) in fp32 (eps 1e-12), rows of a 2-D tensor."""
    _need_cuda(x)
    x = _f32(x)
    out = torch.empty_like(x)
    _cabi.call("cvcl_normalize_rows_f32", _p(x), _p(out), x.shape[0], x.shape[1], _stream())
    return out


@torch.no_grad()
def classify_ncat(img: Tensor, txt: Tensor, normalize: bool = True, log_scale: float = 0.0,
                  want_logits: bool = True) -> Tuple[Tensor, Tensor]:
    """Category classification of frames (the reference's n-category evaluation form,
    multimodal_saycam_data_module.py:545-606 / forward(): logits_per_image = exp(s) * I.T^T, argmax over the C
    category texts).  img [N,E], txt [C,E] features before normalisation.  fp32 end to end.
    -> (pred int32 [N], logits [N,C] | empty)."""
    _need_cuda(img, txt)
    i = normalize_rows_f32(img) if normalize else _f32(img)
    t = normalize_rows_f32(txt) if normalize else _f32(txt)
    scores = linear_f32(i, t, None)                                   # [N, C] cosines
    N, C = scores.shape
    best = torch.empty((N,), dtype=torch.float32, device=img.device)
    pred = torch.empty((N,), dtype=torch.int32, device=img.device)
    _cabi.call("cvcl_row_argmax_f32", _p(scores), C, N, C, 0, 0, _p(best), _p(pred), _stream())
    if not want_logits:
        return pred, scores.new_empty((0,))
    return pred, scores * math.exp(float(log_scale))


def _row_argmax(scores: Tensor) -> Tensor:
    """first maximum of each row of a contiguous [M, N] fp32 matrix (torch.argmax semantics, NaN wins) -> int32 [M]."""
    M, N = scores.shape
    best = torch.empty((M,), dtype=torch.float32, device=scores.device)
    pred = torch.empty((M,), dtype=torch.int32, device=scores.device)
    _cabi.call("cvcl_row_argmax_f32", _p(scores), N, M, N, 0, 0, _p(best), _p(pred), _stream())
    return pred


# ----------------------------------------------------------------------------------------
# spatial-embedding evaluation: fp32 1x1-conv head, spatial "max" / "mean" scores
# ----------------------------------------------------------------------------------------
def _conv_weight(w: Tensor) -> Tensor:
    if w.dim() == 4 and tuple(w.shape[2:]) == (1, 1):
        w = w.reshape(w.shape[0], w.shape[1])
    if w.dim() != 2:
        raise ValueError("conv1x1_f32: weight %s is not [E,K] or [E,K,1,1]" % (tuple(w.shape),))
    return w


@torch.library.custom_op(_NS + "::conv1x1_f32", mutates_args=())
def conv1x1_f32(x: Tensor, w: Tensor, bias: Optional[Tensor]) -> Tensor:
    """The spatial head Conv2d(K, E, 1) (multimodal.py:181-185) in fp32 with fp32 accumulation (cvcl_conv1x1_f32):
    x [B,K,H,W] NCHW layer4 map (read in place), w [E,K] or [E,K,1,1], bias [E] | None -> [B*H*W, E] NHWC rows."""
    w = _conv_weight(w)
    if x.dim() != 4 or x.shape[1] != w.shape[1]:
        raise ValueError("conv1x1_f32: x %s does not fit the weight %s (need x [B,%d,H,W])"
                         % (tuple(x.shape), tuple(w.shape), w.shape[1]))
    if bias is not None and tuple(bias.shape) != (w.shape[0],):
        raise ValueError("conv1x1_f32: bias %s does not fit the weight %s" % (tuple(bias.shape), tuple(w.shape)))
    _need_cuda(x, w, bias)
    x = _f32(x); w = _f32(w)
    bias = _f32(bias) if bias is not None else None
    B, K, H, W = x.shape
    E = w.shape[0]
    out = torch.empty((B * H * W, E), dtype=torch.float32, device=x.device)
    _cabi.call("cvcl_conv1x1_f32", _p(x), _p(w), _p(bias), B, K, H * W, E, _p(out), _stream())
    return out


@conv1x1_f32.register_fake
def _(x, w, bias):
    return x.new_empty((x.shape[0] * x.shape[2] * x.shape[3], w.shape[0]), dtype=torch.float32)


def _location_rows(img: Tensor, normalize: bool) -> Tensor:
    """[M, HW, E] head outputs -> the same as fp32 rows, F.normalize'd per location when `normalize`
    (multimodal.py:736, dim=1 of the NCHW map = the E of each location)."""
    M, HW, E = img.shape
    rows = _f32(img).reshape(M * HW, E)
    return (normalize_rows_f32(rows) if normalize else rows).view(M, HW, E)


def _check_spatial_text(txt: Tensor, lens: Tensor, sim: str, E: int, who: str):
    if sim == "max":
        if txt.dim() != 3 or txt.shape[2] != E:
            raise ValueError("%s: sim='max' takes per-token text features [C, L, %d], got %s" % (who, E, tuple(txt.shape)))
        if lens.dim() != 1 or lens.shape[0] != txt.shape[0]:
            raise ValueError("%s: lens %s does not fit %d labels" % (who, tuple(lens.shape), txt.shape[0]))
    elif sim == "mean":
        if txt.dim() != 2 or txt.shape[1] != E:
            raise ValueError("%s: sim='mean' takes the pooled text factor [C, %d], got %s" % (who, E, tuple(txt.shape)))
    else:
        raise ValueError("%s: sim must be 'max' or 'mean' (got %r)" % (who, sim))


def _spatial_max_scores(rows: Tensor, tok: Tensor, lens: Tensor, txt_index: Optional[Tensor], n_way: int,
                        log_scale: float) -> Tensor:
    M, HW, E = rows.shape
    C, L, _ = tok.shape
    tok = _f32(tok)
    lens = _i64(lens)
    out = torch.empty((M,) if n_way > 0 else (M, C), dtype=torch.float32, device=rows.device)
    _cabi.call("cvcl_spatial_max_scores_f32", _p(rows), _p(tok), _p(lens), _p(txt_index), M, HW, E, C, L, n_way,
               float(log_scale), _p(out), _stream())
    return out


@torch.library.custom_op(_NS + "::eval_nway_spatial", mutates_args=())
def eval_nway_spatial(img: Tensor, txt: Tensor, lens: Tensor, txt_index: Optional[Tensor], n_way: int, sim: str,
                      normalize: bool, log_scale: float, want_logits: bool = True) -> Tuple[Tensor, Tensor]:
    """n-way trials of a spatial-embedding model, fp32 end to end (eval.py:196-214 / multimodal_lit.py:466-511 with
    multimodal.py:757-787).  img [N*n_way, HW, E] head outputs before normalisation (NHWC rows, target first);
    txt: sim="max" per-token text features [C, L, E] (lens [C] their lengths), sim="mean" the pooled text factor
    [C, E] (cvcl_text_encoder_fwd with per_token=1, pool_scale=1/HW); txt_index [N] | None (None: C >= N, trial n
    uses label n).  -> (pred int32 [N], logits = exp(s) * match fp32 [N, n_way] | empty); first maximum wins."""
    if img.dim() != 3 or n_way < 1 or img.shape[0] % n_way != 0:
        raise ValueError("eval_nway_spatial: img %s is not [N*n_way, HW, E] with n_way=%d" % (tuple(img.shape), n_way))
    M, HW, E = img.shape
    N = M // n_way
    _check_spatial_text(txt, lens, sim, E, "eval_nway_spatial")
    if txt_index is not None:
        if tuple(txt_index.shape) != (N,):
            raise ValueError("eval_nway_spatial: txt_index %s does not fit %d trials" % (tuple(txt_index.shape), N))
        txt_index = txt_index.to(torch.int32).contiguous()
    elif txt.shape[0] < N:
        raise ValueError("eval_nway_spatial: %d trials without txt_index need as many labels (got %d)" % (N, txt.shape[0]))
    _need_cuda(img, txt, lens, txt_index)
    rows = _location_rows(img, normalize)
    if sim == "mean":
        # multimodal.py:765-770 factorises: sum over the locations . pooled text / (HW len) -> K7 on the two factors
        return _raw(eval_nway)(_raw(spatial_pool_fwd)(rows), txt, txt_index, n_way, False, log_scale, want_logits)
    logits = _spatial_max_scores(rows, txt, lens, txt_index, n_way, log_scale).view(N, n_way)
    pred = _row_argmax(logits)
    return pred, logits if want_logits else logits.new_empty((0, n_way))


@eval_nway_spatial.register_fake
def _(img, txt, lens, txt_index, n_way, sim, normalize, log_scale, want_logits=True):
    N = img.shape[0] // n_way
    return (img.new_empty((N,), dtype=torch.int32),
            img.new_empty((N, n_way) if want_logits else (0, n_way), dtype=torch.float32))


@torch.library.custom_op(_NS + "::classify_ncat_spatial", mutates_args=())
def classify_ncat_spatial(img: Tensor, txt: Tensor, lens: Tensor, sim: str, normalize: bool, log_scale: float,
                          want_logits: bool = True) -> Tuple[Tensor, Tensor]:
    """Category classification of frames for a spatial-embedding model (multimodal_saycam_data_module.py:545-606 with
    multimodal.py:757-787): img [N, HW, E] head outputs before normalisation, txt / lens as for eval_nway_spatial with
    the C category labels.  -> (pred int32 [N], logits_per_image fp32 [N, C] | empty); first maximum wins."""
    if img.dim() != 3:
        raise ValueError("classify_ncat_spatial: img %s is not [N, HW, E]" % (tuple(img.shape),))
    M, HW, E = img.shape
    _check_spatial_text(txt, lens, sim, E, "classify_ncat_spatial")
    _need_cuda(img, txt, lens)
    rows = _location_rows(img, normalize)
    if sim == "mean":
        return classify_ncat(_raw(spatial_pool_fwd)(rows), txt, False, log_scale, want_logits)
    logits = _spatial_max_scores(rows, txt, lens, None, 0, log_scale)
    pred = _row_argmax(logits)
    return pred, logits if want_logits else logits.new_empty((0,))


@classify_ncat_spatial.register_fake
def _(img, txt, lens, sim, normalize, log_scale, want_logits=True):
    N, C = img.shape[0], txt.shape[0]
    return (img.new_empty((N,), dtype=torch.int32),
            img.new_empty((N, C) if want_logits else (0,), dtype=torch.float32))


@torch.library.custom_op(_NS + "::spatial_attention_f32", mutates_args=())
def spatial_attention_f32(img: Tensor, tok: Tensor, lens: Tensor, text_index: Optional[Tensor], normalize: bool,
                          want_tokens: bool = True) -> Tuple[Tensor, Tensor, Tensor]:
    """Text-to-location attention maps of a spatial-embedding model in fp32 (cvcl_spatial_attention_f32): the
    per-location terms of the spatial similarity (multimodal.py:771-780) before its max / mean reductions.  The
    reference has no function that returns them; they are the summands of its own forward.
    img [M, HW, E] head outputs before normalisation (NHWC rows), normalised per location when `normalize`;
    tok [C, L, E] per-token text features (ops.text_features_spatial, normalised per token iff `normalize`), lens [C];
    text_index [M] picks the label of every image (None: C >= M, image m uses label m).
    -> (token_maps [M, L, HW] | empty, utt_maps [M, HW], token_argmax int32 [M, L] | empty), in match units:
      token_maps[m, l, p] = <x[m, p], tok[c, l]> for l < len[c], exactly 0 past the length;
      utt_maps[m, p] = sum_{l < len} token_maps[m, l, p] / len (len 0 gives NaN); its mean over p is the sim="mean"
      match, and sum_l max_p token_maps[m, l, p] / len is the sim="max" match;
      token_argmax[m, l] = first location of max_p token_maps[m, l, p] (a NaN wins), -1 past the length.
    A text_index outside [0, C) gives NaN maps.  want_tokens=False returns only the utterance maps."""
    if img.dim() != 3:
        raise ValueError("spatial_attention_f32: img %s is not [M, HW, E]" % (tuple(img.shape),))
    M, HW, E = img.shape
    if tok.dim() != 3 or tok.shape[2] != E:
        raise ValueError("spatial_attention_f32: tok %s is not per-token text features [C, L, %d]" % (tuple(tok.shape), E))
    C, L, _ = tok.shape
    if lens.dim() != 1 or lens.shape[0] != C:
        raise ValueError("spatial_attention_f32: lens %s does not fit %d labels" % (tuple(lens.shape), C))
    if text_index is not None:
        if tuple(text_index.shape) != (M,):
            raise ValueError("spatial_attention_f32: text_index %s does not fit %d images" % (tuple(text_index.shape), M))
        text_index = text_index.to(torch.int32).contiguous()
    elif C < M:
        raise ValueError("spatial_attention_f32: %d images without text_index need as many labels (got %d)" % (M, C))
    _need_cuda(img, tok, lens, text_index)
    rows = _location_rows(img, normalize)
    tok = _f32(tok)
    lens = _i64(lens)
    utt = torch.empty((M, HW), dtype=torch.float32, device=img.device)
    if want_tokens:
        maps = torch.empty((M, L, HW), dtype=torch.float32, device=img.device)
        arg = torch.empty((M, L), dtype=torch.int32, device=img.device)
    else:
        maps = utt.new_empty((0,))
        arg = utt.new_empty((0,), dtype=torch.int32)
    _cabi.call("cvcl_spatial_attention_f32", _p(rows), _p(tok), _p(lens), _p(text_index), M, HW, E, C, L,
               _p(maps) if want_tokens else None, _p(utt), _p(arg) if want_tokens else None, _stream())
    return maps, utt, arg


@spatial_attention_f32.register_fake
def _(img, tok, lens, text_index, normalize, want_tokens=True):
    M, HW, _ = img.shape
    L = tok.shape[1]
    return (img.new_empty((M, L, HW) if want_tokens else (0,), dtype=torch.float32),
            img.new_empty((M, HW), dtype=torch.float32),
            img.new_empty((M, L) if want_tokens else (0,), dtype=torch.int32))


@torch.no_grad()
def cosine_nearest(queries: Tensor, keys: Tensor, chunk: int = 16384) -> Tuple[Tensor, Tensor]:
    """Cosine nearest neighbour of every query row among the key rows (analysis_cvcl/duplicates.py:561-607:
    F.normalize + cosine similarity + np.argmax / np.max per evaluation frame).  fp32; the [Nq, Nk] matrix is
    produced in chunks of `chunk` keys and never held whole.  -> (max cosine fp32 [Nq], index int32 [Nq])."""
    _need_cuda(queries, keys)
    q = normalize_rows_f32(queries)
    Nq, Nk = q.shape[0], keys.shape[0]
    best = torch.empty((Nq,), dtype=torch.float32, device=q.device)
    arg = torch.empty((Nq,), dtype=torch.int32, device=q.device)
    for c0 in range(0, Nk, chunk):
        k = normalize_rows_f32(keys[c0:c0 + chunk])
        scores = linear_f32(q, k, None)
        _cabi.call("cvcl_row_argmax_f32", _p(scores), scores.shape[1], Nq, scores.shape[1], c0, int(c0 > 0),
                   _p(best), _p(arg), _stream())
    return best, arg


# ----------------------------------------------------------------------------------------
# cross-modal retrieval: exact top-K, ranks and recall@K in both directions
# ----------------------------------------------------------------------------------------
RETRIEVAL_MAX_K = 64


def check_retrieval_args(n_img: int, n_txt: int, frame_group: Optional[Tensor], text_group: Optional[Tensor],
                         k: int, recall_at, block_bytes: int, who: str = "retrieval_f32"):
    """The argument checks of retrieval_f32, raised as ValueError before any device work."""
    if n_img < 1 or n_txt < 1:
        raise ValueError("%s: needs at least one frame and one text (got %d and %d)" % (who, n_img, n_txt))
    if (frame_group is None) != (text_group is None):
        raise ValueError("%s: frame_group and text_group are given together or not at all" % who)
    if frame_group is None:
        if n_img != n_txt:
            raise ValueError("%s: pair mode (no groups) pairs frame i with text i and needs as many frames as texts "
                             "(got %d and %d)" % (who, n_img, n_txt))
    else:
        for name, grp, n in (("frame_group", frame_group, n_img), ("text_group", text_group, n_txt)):
            if grp.dtype != torch.int64 or tuple(grp.shape) != (n,):
                raise ValueError("%s: %s must be int64 [%d], got %s %s" % (who, name, n, grp.dtype, tuple(grp.shape)))
    kmax = min(RETRIEVAL_MAX_K, n_img, n_txt)
    if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= kmax:
        raise ValueError("%s: k=%r must be an int in [1, min(%d, N_img, N_txt)] = [1, %d]"
                         % (who, k, RETRIEVAL_MAX_K, kmax))
    if any(isinstance(K, bool) or not isinstance(K, int) or K < 1 for K in recall_at):
        raise ValueError("%s: recall_at=%r must hold positive ints" % (who, tuple(recall_at)))
    if isinstance(block_bytes, bool) or not isinstance(block_bytes, int) or block_bytes < 1:
        raise ValueError("%s: block_bytes=%r must be a positive int" % (who, block_bytes))


def _row_blocks(n: int, rows: int, min_rows: int = 1):
    """[q0, q1) blocks of `rows` query rows covering [0, n), every block at least min(min_rows, n) rows long (a
    short tail joins the block before it)."""
    rows = max(rows, min_rows)
    starts = list(range(0, n, rows))
    if len(starts) > 1 and n - starts[-1] < min_rows:
        starts.pop()
    return list(zip(starts, starts[1:] + [n]))


def _retrieval_direction(score_block, n_q: int, n_k: int, q_group, k_group, k: int, scale: Optional[float],
                         block_bytes: int, min_rows: int, dev) -> Tuple[Tensor, Tensor, Tensor]:
    """The query rows in blocks of fp32 scores under block_bytes, each block ranked by cvcl_rank_topk_f32.
    -> (topk, logits = scale * gathered scores (the scores themselves when scale is None), rank)."""
    topk = torch.empty((n_q, k), dtype=torch.int32, device=dev)
    val = torch.empty((n_q, k), dtype=torch.float32, device=dev)
    rank = torch.empty((n_q,), dtype=torch.int32, device=dev)
    for q0, q1 in _row_blocks(n_q, max(1, block_bytes // (4 * n_k)), min_rows):
        s = score_block(q0, q1)
        _cabi.call("cvcl_rank_topk_f32", _p(s), n_k, q1 - q0, n_k, q0, _p(q_group), _p(k_group), k,
                   _p(topk[q0:]), _p(val[q0:]), _p(rank[q0:]), _stream())
        del s
    return topk, (val if scale is None else val * scale), rank


def _retrieval_metrics(rank: Tensor, recall_at) -> Tensor:
    """[recall@K..., mean rank, median rank, n_queries] fp64 on the device, over the queries with a positive;
    ranks 1-based, the median the lower middle value (torch.median)."""
    has = rank >= 0
    n = has.sum()
    nf = n.double()
    recall = torch.stack([(has & (rank < K)).sum() for K in recall_at]).double() / nf if recall_at else nf.new_empty(0)
    mean = ((rank.double() + 1) * has).sum() / nf
    srt = torch.sort(torch.where(has, rank, torch.full_like(rank, 0x7fffffff))).values
    med = srt.gather(0, ((n - 1).clamp(min=0) // 2).view(1)).double() + 1
    med = torch.where(n > 0, med, torch.full_like(med, float("nan")))
    return torch.cat([recall, mean.view(1), med, nf.view(1)])


@torch.no_grad()
def retrieval_f32(img: Tensor, txt: Tensor, lens: Optional[Tensor], sim: str, normalize: bool, log_scale: float,
                  frame_group: Optional[Tensor] = None, text_group: Optional[Tensor] = None, k: int = 10,
                  recall_at=(1, 5, 10), block_bytes: int = 1 << 30) -> dict:
    """Cross-modal retrieval over a held-out split, both directions, exact and fp32 end to end.
    sim="flat":  img [N_img, E] / txt [N_txt, E] features before normalisation (normalised iff `normalize`);
    sim="mean":  img [N_img, HW, E] head outputs (normalised per location iff `normalize`), txt the pooled text
                 factor [N_txt, E];
    sim="max":   img as for "mean", txt per-token text features [N_txt, L, E] with lens [N_txt].
    The scores are the fp32 values classify_ncat / classify_ncat_spatial take their arg-max of: linear_f32 on the
    (normalised) rows for flat, on the pooled factors for mean, cvcl_spatial_max_scores_f32 (exp(s) included) for max.
    Each query row orders the keys as torch.sort(row, descending=True, stable=True): a NaN first, ties by ascending
    key index.  Positives: key i of query i (pair mode, N_img == N_txt), or with frame_group [N_img] / text_group
    [N_txt] (int64) every key whose group equals the query's.  The score blocks hold at most block_bytes of fp32 query
    rows (at least one row; a text->image "max" block at least ceil(64 / L) texts, so that the scores kernel plans
    every block alike and computes the same bits), so the [N_img, N_txt] matrix exists only when it fits.
    -> {"image_to_text": d, "text_to_image": d}, d = {"topk": int32 [Nq, k], "logits": fp32 [Nq, k] (exp(s) * score),
        "rank": int32 [Nq] (0-based position of the first positive, -1 without one), "recall": {K: fraction of the
        queries with a positive whose rank < K}, "mean_rank", "median_rank" (1-based, lower median),
        "n_queries": queries with a positive}.  One device-to-host read, at the end."""
    if sim not in ("flat", "mean", "max"):
        raise ValueError("retrieval_f32: sim must be 'flat', 'mean' or 'max' (got %r)" % (sim,))
    if sim == "flat":
        if img.dim() != 2 or txt.dim() != 2 or img.shape[1] != txt.shape[1]:
            raise ValueError("retrieval_f32: flat features must be img [N_img, E] and txt [N_txt, E], got %s and %s"
                             % (tuple(img.shape), tuple(txt.shape)))
    else:
        if img.dim() != 3:
            raise ValueError("retrieval_f32: img %s is not [N_img, HW, E]" % (tuple(img.shape),))
        _check_spatial_text(txt, lens, sim, img.shape[2], "retrieval_f32")
    recall_at = tuple(recall_at)
    check_retrieval_args(img.shape[0], txt.shape[0], frame_group, text_group, k, recall_at, block_bytes)
    _need_cuda(img, txt, lens if sim == "max" else None, frame_group, text_group)
    fg = _i64(frame_group) if frame_group is not None else None
    tg = _i64(text_group) if text_group is not None else None
    n_img, n_txt = img.shape[0], txt.shape[0]
    min_t2i = 1
    if sim == "max":
        rows = _location_rows(img, normalize)
        tok, lens = _f32(txt), _i64(lens)
        i2t = lambda q0, q1: _spatial_max_scores(rows[q0:q1], tok, lens, None, 0, log_scale)          # noqa: E731
        t2i = lambda q0, q1: _spatial_max_scores(rows, tok[q0:q1], lens[q0:q1], None, 0,               # noqa: E731
                                                 log_scale).t().contiguous()
        min_t2i = -(-RETRIEVAL_MAX_K // tok.shape[1])     # the plan depends on min(texts * L, 64) token rows
        scale = None                                      # the max scores carry exp(s) already
    else:
        if sim == "flat":
            i = normalize_rows_f32(img) if normalize else _f32(img)
            t = normalize_rows_f32(txt) if normalize else _f32(txt)
        else:
            i, t = _raw(spatial_pool_fwd)(_location_rows(img, normalize)), _f32(txt)
        i2t = lambda q0, q1: linear_f32(i[q0:q1], t, None)                                             # noqa: E731
        t2i = lambda q0, q1: linear_f32(t[q0:q1], i, None)                                             # noqa: E731
        scale = math.exp(float(log_scale))
    out, metrics = {}, []
    for name, block, nq, nk, qg, kg, mr in (("image_to_text", i2t, n_img, n_txt, fg, tg, 1),
                                            ("text_to_image", t2i, n_txt, n_img, tg, fg, min_t2i)):
        topk, logits, rank = _retrieval_direction(block, nq, nk, qg, kg, k, scale, block_bytes, mr, img.device)
        out[name] = {"topk": topk, "logits": logits, "rank": rank}
        metrics.append(_retrieval_metrics(rank, recall_at))
    host = torch.stack(metrics).cpu().tolist()
    nr = len(recall_at)
    for name, h in zip(out, host):
        out[name].update(recall={K: h[j] for j, K in enumerate(recall_at)}, mean_rank=h[nr], median_rank=h[nr + 1],
                         n_queries=int(h[nr + 2]))
    return out


# ----------------------------------------------------------------------------------------
# K7 evaluation
# ----------------------------------------------------------------------------------------
@torch.library.custom_op(_NS + "::eval_nway", mutates_args=())
def eval_nway(img: Tensor, txt: Tensor, txt_index: Optional[Tensor], n_way: int, normalize: bool,
              log_scale: float, want_logits: bool = True) -> Tuple[Tensor, Tensor]:
    """img [N*n_way, E] fp32, txt [C,E] fp32, txt_index [N] int32 | None -> (pred [N] i32, logits [N,n_way]).
    want_logits=False returns an empty logits tensor and lets the kernel decide clear-cut trials on raw
    dot products (one division per candidate); near-ties still go through the reference arithmetic, so
    the predictions are the same either way."""
    _need_cuda(img, txt)
    img = _f32(img); txt = _f32(txt)
    E = img.shape[-1]
    N = img.numel() // (E * n_way)
    if txt_index is not None:
        txt_index = txt_index.to(torch.int32).contiguous()
    pred = torch.empty((N,), dtype=torch.int32, device=img.device)
    logits = torch.empty((N, n_way) if want_logits else (0, n_way), dtype=torch.float32, device=img.device)
    _cabi.call("cvcl_eval_nway_fwd", _p(img), _p(txt), _p(txt_index), N, n_way, E, int(normalize),
               float(log_scale), _p(pred), _p(logits) if want_logits else None, _stream())
    return pred, logits


@eval_nway.register_fake
def _(img, txt, txt_index, n_way, normalize, log_scale, want_logits=True):
    N = img.numel() // (img.shape[-1] * n_way)
    return (img.new_empty((N,), dtype=torch.int32),
            img.new_empty((N, n_way) if want_logits else (0, n_way), dtype=torch.float32))


# ----------------------------------------------------------------------------------------
# K6 spatial "max" similarity (multimodal.py:771-780) + InfoNCE on the materialised match
# ----------------------------------------------------------------------------------------
@torch.library.custom_op(_NS + "::spatial_max_fwd", mutates_args=())
def spatial_max_fwd(img16: Tensor, tok16: Tensor, lens: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """img16 [Bi,HW,E] bf16, tok16 [Bt,L,E] bf16 -> (match [Bi,Bt] fp32, amax_it u8, amax_ti u8)."""
    _need_cuda(img16, tok16, lens)
    Bi, HW, E = img16.shape
    Bt, L, _ = tok16.shape
    dev = img16.device
    match = torch.empty((Bi, Bt), dtype=torch.float32, device=dev)
    a_it = torch.empty((Bi, Bt * L), dtype=torch.uint8, device=dev)
    a_ti = torch.empty((Bt * L, Bi), dtype=torch.uint8, device=dev)
    _cabi.call("cvcl_spatial_max_fwd", _p(tok16), _p(img16), _p(_i64(lens)), Bt, L, Bi, HW, E, _p(match),
               _p(a_it), _p(a_ti), _stream())
    return match, a_it, a_ti


@spatial_max_fwd.register_fake
def _(img16, tok16, lens):
    Bi, Bt, L = img16.shape[0], tok16.shape[0], tok16.shape[1]
    return (img16.new_empty((Bi, Bt), dtype=torch.float32), img16.new_empty((Bi, Bt * L), dtype=torch.uint8),
            img16.new_empty((Bt * L, Bi), dtype=torch.uint8))


SPATIAL_MAX_BWD_MMA = True     # False: always use the SIMT gather backward


@torch.library.custom_op(_NS + "::spatial_max_bwd", mutates_args=())
def spatial_max_bwd(g: Tensor, lens: Tensor, ids: Optional[Tensor], a_it: Tensor, a_ti: Tensor,
                    img16: Tensor, tok16: Tensor, need_dimg: bool, need_dtok: bool) -> Tuple[Tensor, Tensor]:
    _need_cuda(g, img16, tok16)
    Bi, HW, E = img16.shape
    Bt, L, _ = tok16.shape
    dev = g.device
    g = _f32(g)
    dimg = torch.empty((Bi, HW, E) if need_dimg else (0,), dtype=torch.float32, device=dev)
    dtok = torch.empty((Bt, L, E) if need_dtok else (0,), dtype=torch.float32, device=dev)
    # tensor-core form (P expansion + two GEMMs) once the problem is big enough to pay for P
    ws = None
    if SPATIAL_MAX_BWD_MMA and Bi * Bt >= 64 * 64:
        nbytes = _cabi.load().cvcl_spatial_max_bwd_workspace_bytes(Bt, L, Bi, HW, E)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    _cabi.call("cvcl_spatial_max_bwd", _p(g), _p(_i64(lens)), None if ids is None else _p(_i64(ids)),
               _p(a_it), _p(a_ti), _p(tok16), _p(img16), Bt, L, Bi, HW, E,
               _p(dtok) if need_dtok else None, _p(dimg) if need_dimg else None, _p(ws), _stream())
    return dimg, dtok


@spatial_max_bwd.register_fake
def _(g, lens, ids, a_it, a_ti, img16, tok16, need_dimg, need_dtok):
    return (g.new_empty(img16.shape if need_dimg else (0,), dtype=torch.float32),
            g.new_empty(tok16.shape if need_dtok else (0,), dtype=torch.float32))


class _SpatialMax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img, tok, lens, ids, split=False):
        Bi, HW, E = img.shape
        Bt, L, _ = tok.shape
        i16, _ = to_bf16_pair(img.reshape(Bi * HW, E), False)
        t16, _ = to_bf16_pair(tok.reshape(Bt * L, E), False)
        i16 = i16.view(Bi, HW, E); t16 = t16.view(Bt, L, E)
        if split and img.dtype == torch.float32 and tok.dtype == torch.float32:
            # scores to fp32 accuracy (hi.hi + lo.hi + hi.lo over a 3E contraction): the arg-max location of
            # near-tied locations agrees with the reference's fp32 einsum; the backward keeps the plain bf16 features
            ic = split_bf16_cat(img.reshape(Bi * HW, E), "hhl").view(Bi, HW, 3 * E)
            tc = split_bf16_cat(tok.reshape(Bt * L, E), "hlh").view(Bt, L, 3 * E)
            match, a_it, a_ti = _raw(spatial_max_fwd)(ic, tc, lens)
        else:
            match, a_it, a_ti = _raw(spatial_max_fwd)(i16, t16, lens)
        ctx.save_for_backward(lens, ids, a_it, a_ti, i16, t16)
        ctx.dt = (img.dtype, tok.dtype)
        return match

    @staticmethod
    def backward(ctx, g):
        lens, ids, a_it, a_ti, i16, t16 = ctx.saved_tensors
        dimg, dtok = _raw(spatial_max_bwd)(g, lens, ids, a_it, a_ti, i16, t16, ctx.needs_input_grad[0],
                                     ctx.needs_input_grad[1])
        return (dimg.to(ctx.dt[0]) if ctx.needs_input_grad[0] else None,
                dtok.to(ctx.dt[1]) if ctx.needs_input_grad[1] else None, None, None, None)


def spatial_max_similarity(img_nhwc, tok, lens, ids=None, split=False):
    """match[i,t] = sum_l max_hw <img[i,hw,:], tok[t,l,:]> / len[t]   (multimodal.py:771-780).
    img_nhwc [Bi,HW,E], tok [Bt,L,E] (fp32 or bf16) -> [Bi,Bt] fp32.  split=True (fp32 inputs): two-term bf16
    operands, scores and arg-max locations to fp32 accuracy at 3x the tensor work."""
    return _SpatialMax.apply(img_nhwc, tok, lens, ids, bool(split))


@torch.library.custom_op(_NS + "::match_infonce_fwd", mutates_args=())
def match_infonce_fwd(match: Tensor, log_scale: float) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    _need_cuda(match)
    match = _f32(match)
    B = match.shape[0]
    if match.shape[1] != B:
        raise ValueError("InfoNCE needs a square similarity matrix, got %s" % (tuple(match.shape),))
    dev = match.device
    lib = _cabi.load()
    ws = torch.empty((lib.cvcl_sim_workspace_bytes(B, B, B, B),), dtype=torch.uint8, device=dev)
    out5 = torch.zeros((8,), dtype=torch.float32, device=dev)
    lse0 = torch.empty((B,), dtype=torch.float32, device=dev); lse1 = torch.empty_like(lse0)
    a0 = torch.empty((B,), dtype=torch.int32, device=dev); a1 = torch.empty_like(a0)
    _cabi.call("cvcl_match_infonce_fwd", _p(match), B, float(log_scale), 1.0 / B, _p(ws), _p(lse0), _p(lse1),
               _p(a0), _p(a1), _p(out5), _stream())
    return out5, lse0, lse1, a0, a1


@match_infonce_fwd.register_fake
def _(match, log_scale):
    B = match.shape[0]
    f = dict(dtype=torch.float32)
    return (match.new_empty((8,), **f), match.new_empty((B,), **f), match.new_empty((B,), **f),
            match.new_empty((B,), dtype=torch.int32), match.new_empty((B,), dtype=torch.int32))


@torch.library.custom_op(_NS + "::match_infonce_bwd", mutates_args=())
def match_infonce_bwd(match: Tensor, log_scale: float, lse0: Tensor, lse1: Tensor) -> Tuple[Tensor, Tensor]:
    _need_cuda(match)
    match = _f32(match)
    B = match.shape[0]
    dmatch = torch.empty_like(match)
    ds = torch.zeros((1,), dtype=torch.float32, device=match.device)
    _cabi.call("cvcl_match_infonce_bwd", _p(match), B, float(log_scale), 0.5 / B, _p(lse0), _p(lse1),
               _p(dmatch), _p(ds), _stream())
    return dmatch, ds


@match_infonce_bwd.register_fake
def _(match, log_scale, lse0, lse1):
    return match.new_empty(match.shape, dtype=torch.float32), match.new_empty((1,), dtype=torch.float32)


class _MatchInfoNCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, match, s):
        ls = _scalar(s)
        out5, lse0, lse1, a0, a1 = _raw(match_infonce_fwd)(match, ls)
        ctx.save_for_backward(match, lse0, lse1)
        ctx.ls = ls
        ctx.s_is_tensor = torch.is_tensor(s)
        ctx.set_materialize_grads(False)          # only the loss is differentiated: no zero gradients for the metrics
        o = out5.unbind(0)
        ctx.mark_non_differentiable(o[1], o[2], o[3], o[4], a0, a1)
        return o[0], o[1], o[2], o[3], o[4], a0, a1

    @staticmethod
    def backward(ctx, gloss, *unused):
        if gloss is None:
            return None, None
        match, lse0, lse1 = ctx.saved_tensors
        dmatch, ds = _raw(match_infonce_bwd)(match, ctx.ls, lse0, lse1)
        return dmatch * gloss, (ds[0] * gloss) if ctx.s_is_tensor and ctx.needs_input_grad[1] else None


def infonce_from_match(match, s):
    """symmetric InfoNCE (multimodal.py:801-818) of logits = exp(s) * match, match [B,B] fp32.
    -> (loss, img_acc, txt_acc, img_ent, txt_ent, logits_per_image, logits_per_text)."""
    loss, iacc, tacc, ient, tent, _, _ = _MatchInfoNCE.apply(match, s)
    with torch.no_grad():
        lpi = match * math.exp(_scalar(s))
    return loss, iacc, tacc, ient, tent, lpi, lpi.t()


# ----------------------------------------------------------------------------------------
# the same loss sharded over a process group: one rank's row block [b,N] and column block [N,b]
# ----------------------------------------------------------------------------------------
def _check_blocks(match_r: Tensor, match_c: Tensor, diag_off: int):
    b, N = match_r.shape
    if tuple(match_c.shape) != (N, b) or not 0 <= diag_off <= N - b:
        raise ValueError("match blocks [b,N] / [N,b] with 0 <= diag_off <= N-b expected, got %s, %s, diag_off=%d"
                         % (tuple(match_r.shape), tuple(match_c.shape), diag_off))
    return b, N


@torch.library.custom_op(_NS + "::match_infonce_block_fwd", mutates_args=())
def match_infonce_block_fwd(match_r: Tensor, match_c: Tensor, diag_off: int, log_scale: float, inv_rows: float
                            ) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """row block [b,N] + column block [N,b] -> (out5 [8] partial sums scaled by inv_rows, lse0 [b], lse1 [b],
    argmax0 [b], argmax1 [b]); positives at (m, m + diag_off) and (m + diag_off, m)."""
    _need_cuda(match_r, match_c)
    match_r = _f32(match_r); match_c = _f32(match_c)
    b, N = _check_blocks(match_r, match_c, diag_off)
    dev = match_r.device
    ws = torch.empty((_cabi.load().cvcl_sim_workspace_bytes(b, N, b, N),), dtype=torch.uint8, device=dev)
    out5 = torch.zeros((8,), dtype=torch.float32, device=dev)
    lse0 = torch.empty((b,), dtype=torch.float32, device=dev); lse1 = torch.empty_like(lse0)
    a0 = torch.empty((b,), dtype=torch.int32, device=dev); a1 = torch.empty_like(a0)
    _cabi.call("cvcl_match_infonce_block_fwd", _p(match_r), _p(match_c), b, N, int(diag_off), float(log_scale),
               float(inv_rows), _p(ws), _p(lse0), _p(lse1), _p(a0), _p(a1), _p(out5), _stream())
    return out5, lse0, lse1, a0, a1


@match_infonce_block_fwd.register_fake
def _(match_r, match_c, diag_off, log_scale, inv_rows):
    b = match_r.shape[0]
    f = dict(dtype=torch.float32)
    return (match_r.new_empty((8,), **f), match_r.new_empty((b,), **f), match_r.new_empty((b,), **f),
            match_r.new_empty((b,), dtype=torch.int32), match_r.new_empty((b,), dtype=torch.int32))


@torch.library.custom_op(_NS + "::match_infonce_block_bwd", mutates_args=())
def match_infonce_block_bwd(match_r: Tensor, match_c: Tensor, diag_off: int, log_scale: float, coef: float,
                            lse0: Tensor, lse1_all: Tensor, lse0_all: Tensor, lse1: Tensor
                            ) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (dmatch_r [b,N], dmatch_c [N,b], dscale [1] of the row block, in a fixed summation order)."""
    _need_cuda(match_r, match_c, lse0, lse1_all, lse0_all, lse1)
    match_r = _f32(match_r); match_c = _f32(match_c)
    b, N = _check_blocks(match_r, match_c, diag_off)
    dev = match_r.device
    ws = torch.empty((_cabi.load().cvcl_match_infonce_block_bwd_workspace_bytes(b, N),), dtype=torch.uint8, device=dev)
    dr = torch.empty_like(match_r); dc = torch.empty_like(match_c)
    ds = torch.empty((1,), dtype=torch.float32, device=dev)
    _cabi.call("cvcl_match_infonce_block_bwd", _p(match_r), _p(match_c), b, N, int(diag_off), float(log_scale),
               float(coef), _p(_f32(lse0)), _p(_f32(lse1_all)), _p(_f32(lse0_all)), _p(_f32(lse1)), _p(dr), _p(dc),
               _p(ds), _p(ws), _stream())
    return dr, dc, ds


@match_infonce_block_bwd.register_fake
def _(match_r, match_c, diag_off, log_scale, coef, lse0, lse1_all, lse0_all, lse1):
    f = dict(dtype=torch.float32)
    return match_r.new_empty(match_r.shape, **f), match_c.new_empty(match_c.shape, **f), match_r.new_empty((1,), **f)


def _spatial_max_block_fwd(split):
    """The CUDA arithmetic of sharding.spatial_max_infonce_forward: both blocks through spatial_max_fwd, then the block
    InfoNCE statistics.  The gathered features are fp32 (split: the two-term operands and the bf16 backward operands
    are built here, exactly as the one-device _SpatialMax builds them for the same pairs) or already bf16."""
    def fwd_operand(x, pattern):
        n, k, E = x.shape
        if split:
            return split_bf16_cat(x.reshape(n * k, E), pattern).view(n, k, 3 * E)
        return x

    def bf16(x):
        n, k, E = x.shape
        return to_bf16_pair(x.reshape(n * k, E), False)[0].view(n, k, E)

    def compute(img_r, tok_r, lens_r, ids_r, img_all, tok_all, lens_all, ids_all, ls, diag_off, inv_rows):
        fwd = _raw(spatial_max_fwd)
        match_r, ait_r, ati_r = fwd(fwd_operand(img_r, "hhl"), fwd_operand(tok_all, "hlh"), lens_all)
        match_c, ait_c, ati_c = fwd(fwd_operand(img_all, "hhl"), fwd_operand(tok_r, "hlh"), lens_r)
        out5, lse0, lse1, a0, a1 = _raw(match_infonce_block_fwd)(match_r, match_c, diag_off, ls, inv_rows)
        state = (match_r, match_c, ait_r, ati_r, ait_c, ati_c, bf16(img_r), bf16(tok_r), bf16(img_all), bf16(tok_all),
                 lens_r, ids_r, lens_all, ids_all, ls)
        return out5, lse0, lse1, a0, a1, state
    return compute


def _spatial_max_block_bwd(state, diag_off, coef, lse0, lse1_all, lse0_all, lse1):
    (match_r, match_c, ait_r, ati_r, ait_c, ati_c, i16_r, t16_r, i16_all, t16_all,
     lens_r, ids_r, lens_all, ids_all, ls) = state
    g_r, g_c, ds = _raw(match_infonce_block_bwd)(match_r, match_c, diag_off, ls, coef, lse0, lse1_all, lse0_all, lse1)
    bwd = _raw(spatial_max_bwd)
    dimg, _ = bwd(g_r, lens_all, ids_all, ait_r, ati_r, i16_r, t16_all, True, False)
    del g_r
    _, dtok = bwd(g_c, lens_r, ids_r, ait_c, ati_c, i16_all, t16_r, False, True)
    return dimg, dtok, ds


class _SpatialMaxInfoNCE(torch.autograd.Function):
    """spatial_max_similarity + infonce_from_match with the batch sharded over a process group (sharding.py): the
    location and token features are all-gathered, each rank evaluates its row block and column block of the match
    matrix.  Same outputs and gradient contract as _SimInfoNCE: the five scalars and d s are global on every rank,
    d img / d tok are for the local pairs.  The eighth output is the rank's own [b,b] block of the match matrix."""

    @staticmethod
    def forward(ctx, img, tok, lens, ids, s, group, split):
        from . import sharding
        split = bool(split) and img.dtype == torch.float32 and tok.dtype == torch.float32
        if split:
            gi, gt = img.detach(), tok.detach()
        else:
            gi = to_bf16_pair(img.reshape(-1, img.shape[-1]), False)[0].view(img.shape)
            gt = to_bf16_pair(tok.reshape(-1, tok.shape[-1]), False)[0].view(tok.shape)
        out5, saved, (a0, a1) = sharding.spatial_max_infonce_forward(gi, gt, lens, ids, _scalar(s), group,
                                                                     _spatial_max_block_fwd(split))
        ctx.saved = saved
        ctx.group = group
        ctx.meta = (img.dtype, tok.dtype, torch.is_tensor(s))
        ctx.set_materialize_grads(False)          # only the loss is differentiated: no zero gradients for the metrics
        state, _, _, rank, b = saved[:5]
        local = state[0][:, rank * b:(rank + 1) * b].clone()      # match_r restricted to this rank's texts
        o = out5[:5].unbind(0)
        ctx.mark_non_differentiable(o[1], o[2], o[3], o[4], a0, a1, local)
        return o[0], o[1], o[2], o[3], o[4], a0, a1, local

    @staticmethod
    def backward(ctx, gloss, *unused):
        from . import sharding
        if gloss is None:
            return None, None, None, None, None, None, None
        idt, tdt, s_is_tensor = ctx.meta
        dimg, dtok, ds = sharding.spatial_max_infonce_backward(ctx.saved, ctx.group, _spatial_max_block_bwd)
        dimg = (dimg * gloss).to(idt)
        dtok = (dtok * gloss).to(tdt)
        ds_out = (ds[0] * gloss) if (s_is_tensor and ctx.needs_input_grad[4]) else None
        return dimg, dtok, None, None, ds_out, None, None


def spatial_max_infonce(img_nhwc, tok, lens, ids, s, group=None, split=False, local_match=False):
    """symmetric InfoNCE of the spatial "max" similarity (multimodal.py:771-822) with the batch sharded over `group`:
    img_nhwc [b,HW,E] and tok [b,L,E] (fp32, or bf16) are this rank's pairs; ranks may hold different L.
    -> (loss, image_accuracy, text_accuracy, image_entropy, text_entropy, image_pred, text_pred), all global but the
    two arg-max vectors (this rank's images / texts, indices into the global batch); local_match=True appends the
    rank's own [b,b] block of the match matrix.  split=True: two-term bf16 operands for the scores (see
    spatial_max_similarity).  Gradients: d img / d tok for the local pairs, d s global; replicated parameters get
    local partials to be summed with sharding.allreduce_gradients."""
    out = _SpatialMaxInfoNCE.apply(img_nhwc, tok, lens, ids, s, group, bool(split))
    return out if local_match else out[:7]


# ----------------------------------------------------------------------------------------
# Grad-CAM attention maps (SURVEY 8f item 4; multimodal/attention_maps.py:111-165)
# ----------------------------------------------------------------------------------------
@torch.library.custom_op(_NS + "::gradcam_flat", mutates_args=())
def gradcam_flat(act: Tensor, w: Tensor, bias: Optional[Tensor], target: Tensor, normalize: bool) -> Tensor:
    """act [N,K,H,W] fp32 layer4 activation, w [E,K], bias [E] | None, target [N,E] -> cam [N,1,H,W] fp32
    = clamp(sum_c act * alpha, 0) with alpha the spatial mean of d<normalize(fc(avgpool(act))), target>/d act
    (closed form: the head is linear in the pooled activation, no trunk backward)."""
    _need_cuda(act, w, target)
    act = _f32(act); w = _f32(w); target = _f32(target)
    bias = None if bias is None else _f32(bias)
    N, K, H, W = act.shape
    E = w.shape[0]
    if w.shape[1] != K or tuple(target.shape) != (N, E):
        raise ValueError("gradcam_flat: act %s, w %s, target %s do not fit" % (tuple(act.shape), tuple(w.shape),
                                                                              tuple(target.shape)))
    lib = _cabi.load()
    ws = torch.empty((max(int(lib.cvcl_gradcam_workspace_bytes(N, K, E)), 16),), dtype=torch.uint8, device=act.device)
    cam = torch.empty((N, 1, H, W), dtype=torch.float32, device=act.device)
    _cabi.call("cvcl_gradcam_flat", _p(act), _p(w), _p(bias), _p(target), N, K, H * W, E, int(normalize), _p(ws),
               _p(cam), _stream())
    return cam


@gradcam_flat.register_fake
def _(act, w, bias, target, normalize):
    N, K, H, W = act.shape
    return act.new_empty((N, 1, H, W), dtype=torch.float32)


@torch.library.custom_op(_NS + "::bicubic_upsample", mutates_args=())
def bicubic_upsample(x: Tensor, out_h: int, out_w: int) -> Tensor:
    """x [N,1,h,w] fp32 -> [N,1,out_h,out_w]: F.interpolate(mode="bicubic", align_corners=False)."""
    _need_cuda(x)
    x = _f32(x)
    N, C, h, w = x.shape
    out = torch.empty((N, C, out_h, out_w), dtype=torch.float32, device=x.device)
    _cabi.call("cvcl_bicubic_upsample", _p(x), N * C, h, w, int(out_h), int(out_w), _p(out), _stream())
    return out


@bicubic_upsample.register_fake
def _(x, out_h, out_w):
    return x.new_empty((x.shape[0], x.shape[1], out_h, out_w), dtype=torch.float32)
