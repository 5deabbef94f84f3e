"""Global-batch InfoNCE sharded by pairs over the ranks of a torch.distributed group
(SURVEY section 8e; the reference itself is single-process -- its oracle for this path is the
single-process loss on the concatenated batch).

Rank r owns pairs [r*b, (r+1)*b).  One exchange step: all-gather of the L2-normalised bf16
features.  Each rank then evaluates its ROW block  S[R, :] = e^s I_R T_all^T  (image->text CE of
its b images) and its COLUMN block  S[:, R]^T = e^s T_R I_all^T  (text->image CE of its b texts);
the positives sit at column offset r*b.  Backward: all-gather the 2*B fp32 log-sum-exps, then
  dI_R = e^s G[R, :] T_all,   dT_R = e^s G[:, R]^T I_all,   G = (P_row + P_col - 2 I) / (2B)
so no reduce-scatter of feature gradients is needed; d s is all-reduced.  The spatial "max" similarity shards the
same way on its materialised match blocks (`spatial_max_infonce_forward` / `_backward`).

The collectives live here; the arithmetic is injected (`compute_fwd` / `compute_bwd`): the
product passes the CUDA ops of `ops.py`, the CPU (gloo) tests pass a torch restatement so the
orchestration (offsets, gathers, reductions) is covered without a GPU.
"""
from __future__ import annotations

import os

import torch
import torch.distributed as dist


def group_info(group):
    if group is None or not dist.is_available() or not dist.is_initialized():
        return 1, 0
    return dist.get_world_size(group), dist.get_rank(group)


def all_gather_rows(t: torch.Tensor, group, world: int) -> torch.Tensor:
    """[b, ...] per rank -> [world*b, ...] in rank order (identity when world == 1)."""
    if world == 1:
        return t
    out = torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, t.contiguous(), group=group)
    return out


def infonce_forward(img, txt, log_scale, group, compute_fwd):
    """img, txt: local [b, E] operands.  Returns (out5 global [>=5], saved-for-backward tuple,
    local argmax pair)."""
    world, rank = group_info(group)
    b = img.shape[0]
    img_all = all_gather_rows(img, group, world)
    txt_all = all_gather_rows(txt, group, world)
    Bg = world * b
    out5, lse0, lse1, a0, a1 = compute_fwd(img, txt_all, txt, img_all, log_scale, rank * b, 1.0 / Bg)
    out5 = out5.clone()
    if world > 1:
        dist.all_reduce(out5, group=group)       # partial sums already scaled by 1/B_global
    saved = (img, txt, img_all, txt_all, lse0, lse1, log_scale, rank, b, world)
    return out5, saved, (a0, a1)


def infonce_backward(saved, group, compute_bwd):
    """-> (dimg [b,E], dtxt [b,E], dscale [1]) for upstream gradient 1."""
    img, txt, img_all, txt_all, lse0, lse1, log_scale, rank, b, world = saved
    lse0_all = all_gather_rows(lse0, group, world)
    lse1_all = all_gather_rows(lse1, group, world)
    Bg = world * b
    dimg, dtxt, ds = compute_bwd(img, txt_all, txt, img_all, log_scale, rank * b, 0.5 / Bg,
                                 lse0, lse1_all, lse1, lse0_all)
    if world > 1:
        dist.all_reduce(ds, group=group)
    return dimg, dtxt, ds


def spatial_max_infonce_forward(img, tok, lens, ids, log_scale, group, compute_fwd, pad_id=0):
    """Spatial "max" InfoNCE sharded by pairs (same row / column decomposition as `infonce_forward`).

    img [b, HW, ...] location features, tok [b, L, ...] per-token features, lens [b], ids [b, L] (or None) of this
    rank's pairs; the feature tensors are gathered as given (fp32 or bf16: the caller chooses).  Ranks may hold
    different L (the collate pads to each batch's longest utterance): one all-gather of (b, L) finds the longest,
    and every rank pads its tokens with zero rows and its ids with `pad_id` to that length before the gathers --
    positions beyond len[t] do not enter match[i, t].  A rank count b that differs between ranks raises the same
    ValueError on every rank (the gathers need equal blocks).

    compute_fwd(img_r, tok_r, lens_r, ids_r, img_all, tok_all, lens_all, ids_all, log_scale, diag_off, inv_rows)
      -> (out5, lse0 [b], lse1 [b], argmax0 [b], argmax1 [b], state)
    evaluates the row block spatial_max(img_r, tok_all) [b, N] and the column block spatial_max(img_all, tok_r)
    [N, b].  Returns (out5 global, saved-for-backward tuple, local argmax pair)."""
    world, rank = group_info(group)
    b, L = tok.shape[0], tok.shape[1]
    if img.shape[0] != b or lens.shape[0] != b:
        raise ValueError("spatial max InfoNCE: %d images, %d texts and %d lengths on rank %d"
                         % (img.shape[0], b, lens.shape[0], rank))
    sizes = all_gather_rows(torch.tensor([[b, L]], dtype=torch.int64, device=img.device), group, world)
    bs, Ls = sizes[:, 0].tolist(), sizes[:, 1].tolist()
    if len(set(bs)) != 1:
        raise ValueError("sharded spatial max InfoNCE needs the same number of pairs on every rank, got %s" % (bs,))
    Lm = max(Ls)
    if Lm > L:
        tok = torch.cat([tok, tok.new_zeros((b, Lm - L) + tuple(tok.shape[2:]))], dim=1)
        if ids is not None:
            ids = torch.cat([ids, ids.new_full((b, Lm - L), pad_id)], dim=1)
    img_all = all_gather_rows(img, group, world)
    tok_all = all_gather_rows(tok, group, world)
    lens_all = all_gather_rows(lens, group, world)
    ids_all = None if ids is None else all_gather_rows(ids, group, world)
    Bg = world * b
    out5, lse0, lse1, a0, a1, state = compute_fwd(img, tok, lens, ids, img_all, tok_all, lens_all, ids_all,
                                                  log_scale, rank * b, 1.0 / Bg)
    out5 = out5.clone()
    if world > 1:
        dist.all_reduce(out5, group=group)       # partial sums already scaled by 1/B_global
    saved = (state, lse0, lse1, rank, b, world, L)
    return out5, saved, (a0, a1)


def spatial_max_infonce_backward(saved, group, compute_bwd):
    """-> (dimg [b, HW, E], dtok [b, L, E] at this rank's own L, dscale [1] summed over the ranks) for upstream
    gradient 1.  compute_bwd(state, diag_off, coef, lse0, lse1_all, lse0_all, lse1) -> (dimg, dtok, ds of the row
    block).  Each image's row and each text's column live on its own rank: no reduce-scatter."""
    state, lse0, lse1, rank, b, world, L = saved
    lse0_all = all_gather_rows(lse0, group, world)
    lse1_all = all_gather_rows(lse1, group, world)
    dimg, dtok, ds = compute_bwd(state, rank * b, 0.5 / (world * b), lse0, lse1_all, lse0_all, lse1)
    if world > 1:
        dist.all_reduce(ds, group=group)
    return dimg, (dtok if dtok.shape[1] == L else dtok[:, :L].contiguous()), ds


def allreduce_gradients(params, group=None):
    """Sum the per-rank partial gradients of replicated parameters (head weight/bias, embedding
    table): the loss is the GLOBAL-batch loss on every rank, so the correct reduction is SUM, not
    the mean a DDP wrapper would apply.  One flat all-reduce (about 9 MB for CVCL)."""
    world, _ = group_info(group)
    grads = [p.grad for p in params if p.grad is not None]
    if world == 1 or not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, group=group)
    off = 0
    for g in grads:
        n = g.numel()
        g.copy_(flat[off:off + n].view_as(g))
        off += n


# ----------------------------------------------------------------------------------------------
# exchange + gradient sum over NVLink peer memory (symmetric memory) instead of NCCL collectives
# ----------------------------------------------------------------------------------------------
def _align(n, a=256):
    return (n + a - 1) // a * a


class PeerExchange:
    """Per-(group, b, E, n_stats) symmetric-memory arena for the three collectives of the sharded step:

        [ feats (b, 2E) bf16 | lse (2, b) f32 | feats_all (W*b, 2E) | lse_all (2, W*b) | reduce scratch |
          stats (n_stats) f32 x N_SLOTS | flags ]

    is allocated once in peer-mapped memory (one rendezvous); each collective is ONE kernel of
    `csrc/peer_collectives.cuh` that carries its own cross-rank barrier (flag words written over
    NVLink) -- `cvcl_peer_allgather` for the features and the LSEs, `cvcl_peer_allreduce_f32` (two-shot,
    in place, deterministic) for [out5 | ds | db | dtable | dW] -- instead of two NCCL all-gathers and
    an NCCL all-reduce.  Default: the PUSH kernels (posted stores over NVLink, no load round trips;
    CVCL_B200_PEER_MODE=pull selects the pull kernels).  Reuse across steps is safe because a rank overwrites its blocks for step s+1
    only after the all-reduce (or the closing barrier) of step s, which no rank leaves before every
    rank has finished reading step s.  Default on when symmetric memory is available;
    CVCL_B200_SYMM=0 selects the NCCL collectives."""

    _cache = {}
    CH_FEATS, CH_LSE, CH_REDUCE, CH_BARRIER, CH_FUSED = 0, 1, 2, 3, 4
    N_SLOTS = 2          # stats blocks: alternating CUDA graphs keep the previous step's gradients readable

    def __init__(self, group, b, E, n_stats, dev, min_scratch=0):
        import ctypes
        import torch.distributed._symmetric_memory as symm
        from . import _cabi
        lib = _cabi.load()
        self.world, self.rank = group_info(group)
        self.b, self.E, self.n_stats = b, E, n_stats
        self.timeout_ms = int(os.environ.get("CVCL_B200_PEER_TIMEOUT_MS", "600000"))
        fw = int(lib.cvcl_peer_flag_words())
        nblk = int(lib.cvcl_peer_max_blocks())
        self.push = os.environ.get("CVCL_B200_PEER_MODE", "push") != "pull"
        Bg = self.world * b
        sizes = [("feats", b * 2 * E * 2), ("lse", 2 * b * 4), ("feats_all", Bg * 2 * E * 2), ("lse_all", 2 * Bg * 4),
                 ("scratch", max(int(lib.cvcl_peer_allreduce_scratch_bytes(n_stats, self.world)), int(min_scratch)))]
        # gathered features of the one-kernel sharded step (texts and images separately: each is the key operand of
        # one direction) and a fifth flag channel for its in-kernel cross-rank barriers
        part_bytes = int(lib.cvcl_flat_fused_sharded_part_bytes(b, self.world))
        sizes += [("txt_all", Bg * E * 2), ("img_all", Bg * E * 2), ("part_all", part_bytes)]
        sizes += [("stats%d" % k, n_stats * 4) for k in range(self.N_SLOTS)] + [("flags", 5 * fw * 4)]
        off, total = {}, 0
        for name, nb in sizes:
            off[name] = total
            total += _align(nb)
        self.arena = symm.empty((total,), dtype=torch.uint8, device=dev)
        self.arena.zero_()
        self.handle = symm.rendezvous(self.arena, group)
        torch.cuda.synchronize(dev)
        dist.barrier(group=group)            # every rank's flag words are zero before anyone signals
        torch.cuda.synchronize(dev)

        def view(name, nbytes, dtype):
            return self.arena[off[name]:off[name] + nbytes].view(dtype)
        self.feats = view("feats", b * 2 * E * 2, torch.bfloat16).view(b, 2 * E)
        self.lse = view("lse", 2 * b * 4, torch.float32).view(2, b)
        self.feats_all = view("feats_all", Bg * 2 * E * 2, torch.bfloat16).view(Bg, 2 * E)
        self.lse_all = view("lse_all", 2 * Bg * 4, torch.float32).view(2, Bg)
        self.stats = [view("stats%d" % k, n_stats * 4, torch.float32) for k in range(self.N_SLOTS)]
        self.epoch = torch.zeros((4, nblk), dtype=torch.int32, device=dev)
        self.status = torch.zeros((1,), dtype=torch.int32, device=dev)
        ptrs = [int(p) for p in self.handle.buffer_ptrs]
        arr = ctypes.c_void_p * self.world

        def table(name, extra=0):
            return arr(*[p + off[name] + extra for p in ptrs])
        self.p_feats, self.p_lse = table("feats"), table("lse")
        self.p_feats_all, self.p_lse_all, self.p_scratch = table("feats_all"), table("lse_all"), table("scratch")
        self.p_stats = [table("stats%d" % k) for k in range(self.N_SLOTS)]
        self.p_flags = [table("flags", ch * fw * 4) for ch in range(5)]
        self.txt_all = view("txt_all", Bg * E * 2, torch.bfloat16).view(Bg, E)
        self.img_all = view("img_all", Bg * E * 2, torch.bfloat16).view(Bg, E)
        self.p_txt_all, self.p_img_all, self.p_part_all = table("txt_all"), table("img_all"), table("part_all")
        self.fused_epoch = torch.zeros((1,), dtype=torch.int32, device=dev)
        self._self_test(group, dev)

    NO_TRAP = 0x80000000

    def _self_test(self, group, dev):
        """Run every collective twice on known patterns with a short, non-trapping timeout and compare on
        every rank; all ranks agree (NCCL all-reduce of the verdict) or the exchange is rejected and the
        step keeps the NCCL collectives.  Costs a few hundred microseconds once per (group, shape)."""
        st = torch.cuda.current_stream(dev).cuda_stream
        keep, self.timeout_ms = self.timeout_ms, 3000 | self.NO_TRAP
        W, r, b, E, n = self.world, self.rank, self.b, self.E, self.n_stats
        ok = True
        try:
            for it in (1, 2):
                col = torch.arange(2 * E, device=dev, dtype=torch.float32) % 7
                self.feats.copy_((col[None, :] + (r + it)).expand(b, 2 * E))
                self.lse.copy_(torch.arange(2 * b, device=dev, dtype=torch.float32).view(2, b) + 1000.0 * (r + it))
                base = (torch.arange(n, device=dev, dtype=torch.float32) % 13) - 6.0
                for k in range(self.N_SLOTS):
                    self.stats[k].copy_(base * (r + 1 + k))
                # copies are taken BEFORE the closing barrier in stream order: a faster rank may start the
                # next round (and push into this rank's gathered buffers) as soon as it has passed it
                fa = self.gather_feats(st).clone()
                la = self.gather_lse(st).clone()
                for k in range(self.N_SLOTS):
                    self.allreduce_stats(k, n, st)
                got = [self.stats[k].clone() for k in range(self.N_SLOTS)]
                self.barrier(st)
                torch.cuda.synchronize(dev)
                want_f = torch.cat([(col[None, :] + (q + it)).expand(b, 2 * E) for q in range(W)]).to(torch.bfloat16)
                want_l = torch.cat([torch.arange(2 * b, device=dev, dtype=torch.float32).view(2, b) + 1000.0 * (q + it)
                                    for q in range(W)], dim=1)
                ok = ok and torch.equal(fa, want_f) and torch.equal(la, want_l)
                for k in range(self.N_SLOTS):
                    ok = ok and torch.equal(got[k], base * float(sum(q + 1 + k for q in range(W))))
            ok = ok and int(self.status.item()) == 0
        except Exception:                        # noqa: BLE001
            ok = False
        verdict = torch.tensor([1 if ok else 0], device=dev, dtype=torch.int32)
        dist.all_reduce(verdict, op=dist.ReduceOp.MIN, group=group)
        self.timeout_ms = keep
        if int(verdict.item()) != 1:
            raise RuntimeError("peer-memory collectives failed their start-up self-test on this machine")
        for k in range(self.N_SLOTS):
            self.stats[k].zero_()
        torch.cuda.synchronize(dev)
        dist.barrier(group=group)

    @classmethod
    def get(cls, group, b, E, n_stats, dev, min_scratch=0):
        if os.environ.get("CVCL_B200_SYMM", "1") == "0":
            return None
        world, _ = group_info(group)
        if world not in (2, 4, 8) or b % 4 or n_stats % 4 or (b * 2 * E * 2) % 16:
            return None
        # keyed by the group's identity (name + ranks), not id(): a destroyed group's id can be recycled
        try:
            gkey = (dist.get_process_group_ranks(group).__repr__(), getattr(group, "group_name", ""))
        except Exception:                        # noqa: BLE001
            gkey = id(group)
        key = (gkey, b, E, n_stats, dev.index, os.environ.get("CVCL_B200_PEER_MODE", "push"), int(min_scratch))
        if key not in cls._cache:
            try:
                cls._cache[key] = cls(group, b, E, n_stats, dev, min_scratch)
            except Exception as exc:             # noqa: BLE001  (no symmetric memory / failed self-test)
                import warnings
                warnings.warn("cvcl_b200: peer-memory exchange unavailable (%r); using the NCCL collectives" % (exc,))
                cls._cache[key] = None
        return cls._cache[key]

    def _ep(self, ch):
        return self.epoch[ch].data_ptr()

    def gather_feats(self, stream):
        """-> [world*b, 2E] bf16: every rank's [img|txt] feature block (persistent symmetric buffer)."""
        from . import _cabi
        nbytes = self.b * 2 * self.E * 2
        ch = self.CH_FEATS
        if self.push:
            _cabi.call("cvcl_peer_allgather_push", self.p_feats_all, self.p_flags[ch], self._ep(ch),
                       self.status.data_ptr(), self.world, self.rank, self.feats.data_ptr(), nbytes, 1, 0, 0,
                       self.timeout_ms, stream)
        else:
            _cabi.call("cvcl_peer_allgather", self.p_feats, self.p_flags[ch], self._ep(ch), self.status.data_ptr(),
                       self.world, self.rank, nbytes, 1, 0, self.feats_all.data_ptr(), 0, self.timeout_ms, stream)
        return self.feats_all

    def gather_lse(self, stream):
        """-> [2, world*b] fp32: every rank's lse0 / lse1."""
        from . import _cabi
        nb = self.b * 4
        ch = self.CH_LSE
        if self.push:
            _cabi.call("cvcl_peer_allgather_push", self.p_lse_all, self.p_flags[ch], self._ep(ch),
                       self.status.data_ptr(), self.world, self.rank, self.lse.data_ptr(), nb, 2, nb, self.world * nb,
                       self.timeout_ms, stream)
        else:
            _cabi.call("cvcl_peer_allgather", self.p_lse, self.p_flags[ch], self._ep(ch), self.status.data_ptr(),
                       self.world, self.rank, nb, 2, nb, self.lse_all.data_ptr(), self.world * nb, self.timeout_ms,
                       stream)
        return self.lse_all

    def allreduce_stats(self, slot, n, stream):
        """in-place sum over ranks of the first n floats of stats block `slot`."""
        from . import _cabi
        ch = self.CH_REDUCE
        if self.push:
            _cabi.call("cvcl_peer_allreduce_push_f32", self.p_stats[slot], self.p_scratch, self.p_flags[ch],
                       self._ep(ch), self.status.data_ptr(), self.world, self.rank, n, self.timeout_ms, stream)
        else:
            _cabi.call("cvcl_peer_allreduce_f32", self.p_stats[slot], self.p_flags[ch], self._ep(ch),
                       self.status.data_ptr(), self.world, self.rank, n, self.timeout_ms, stream)

    def barrier(self, stream):
        from . import _cabi
        _cabi.call("cvcl_peer_barrier", self.p_flags[self.CH_BARRIER], self._ep(self.CH_BARRIER),
                   self.status.data_ptr(), self.world, self.rank, self.timeout_ms, stream)

    def check(self):
        """raise if a cross-rank barrier timed out (synchronises the device)."""
        if int(self.status.item()) != 0:
            raise RuntimeError("peer collective barrier timed out (status %d)" % int(self.status.item()))
