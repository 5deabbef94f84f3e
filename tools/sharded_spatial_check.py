"""torchrun target: the spatial "max" contrastive loss sharded over a process group == the single-GPU result on the
concatenated batch, for both spatial_max_precision modes, with a different utterance length L on every rank.
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/sharded_spatial_check.py [b]
(1) op level: ops.spatial_max_infonce (loss, metrics, d img, d tok, d s) against spatial_max_similarity +
infonce_from_match on the whole batch; (2) the model step through MultiModalModel.calculate_contrastive_loss +
backward() + sharding.allreduce_gradients (fix_temperature) against the single-GPU step; (3) with more than one rank,
unequal pair counts raise ValueError on every rank.  Prints `SHARDED_SPATIAL_OK ...` on rank 0, raises otherwise."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); lr = int(os.environ["LOCAL_RANK"])
dev = torch.device("cuda", lr); torch.cuda.set_device(dev)
dist.init_process_group("nccl", device_id=dev)
import multimodal_baby_b200 as m
from oracle import cvcl_oracle as O
from oracle.make_golden import case_inputs

G = dist.group.WORLD
E, V, HW = 512, 2350, 49
S = float(-np.log(0.07))
b = int(sys.argv[1]) if len(sys.argv) > 1 else 48
B = world * b
sl = slice(rank * b, (rank + 1) * b)
Ls = [25 - 3 * r for r in range(world)]                      # every rank's batch padded to its own longest utterance
Lr, Lm = Ls[rank], max(Ls)


def rel(a, c):
    return float((a - c).norm() / c.norm())


def tokens(seed):
    """ids [B, Lm], lens [B]: rank r's rows are a collate batch of longest utterance Ls[r], padded to Lm"""
    rng = np.random.RandomState(seed)
    ids = np.zeros((B, Lm), np.int64); lens = np.zeros(B, np.int64)
    for r in range(world):
        i, n = O.synth_tokens(rng, b, Ls[r], V)
        n[0] = Ls[r]; i[0, :] = 5; i[0, 0] = 2; i[0, Ls[r] - 1] = 3
        ids[r * b:(r + 1) * b, :Ls[r]] = i; lens[r * b:(r + 1) * b] = n
    return torch.from_numpy(ids).to(dev), torch.from_numpy(lens).to(dev)


def build(group, inp, precision):
    args = argparse.Namespace(embedding_type="spatial", embedding_dim=E, normalize_features=True, fix_temperature=True,
                              temperature=0.07, text_encoder="embedding", sim="max")
    vocab = {str(i): i for i in range(V)}
    model = m.MultiModalModel(m.VisionEncoder(args, trunk="pooled"), m.TextEncoder(vocab, 2048, args), args)
    with torch.no_grad():
        conv = model.image_embed.model[-1]
        conv.weight.copy_(torch.from_numpy(inp["W"])[:, :, None, None]); conv.bias.copy_(torch.from_numpy(inp["b"]))
        model.text_embed.embedding.weight.copy_(torch.from_numpy(inp["table"]))
    model.process_group = group
    model.spatial_max_precision = precision
    return model.to(dev).train()


for precision in ("split_bf16", "bf16"):
    split = precision == "split_bf16"
    # (1) op level, s differentiated
    ids, lens = tokens(7)
    gen = torch.Generator().manual_seed(7)
    img = torch.nn.functional.normalize(torch.randn(B, HW, E, generator=gen), dim=-1).to(dev)
    tok = torch.nn.functional.normalize(torch.randn(B, Lm, E, generator=gen), dim=-1).to(dev)
    tok = tok * (torch.arange(Lm, device=dev)[None, :] < lens[:, None])[..., None]

    def one_gpu():
        i = img.clone().requires_grad_(True); t = tok.clone().requires_grad_(True)
        s = torch.tensor(S, device=dev, requires_grad=True)
        out = m.ops.infonce_from_match(m.ops.spatial_max_similarity(i, t, lens, ids, split=split), s)
        out[0].backward()
        return [o.detach() for o in out[:5]], i.grad, t.grad, s.grad
    r5, rdi, rdt, rds = one_gpu()
    i = img[sl].clone().requires_grad_(True); t = tok[sl, :Lr].clone().requires_grad_(True)
    s = torch.tensor(S, device=dev, requires_grad=True)
    out = m.ops.spatial_max_infonce(i, t, lens[sl], ids[sl, :Lr], s, G, split=split)
    out[0].backward()
    for k in range(5):
        a, c = r5[k].item(), out[k].item()
        assert abs(a - c) <= 2e-6 * max(1.0, abs(a)), (precision, k, a, c)
    assert rel(i.grad, rdi[sl]) <= 1e-5, (precision, rel(i.grad, rdi[sl]))
    assert rel(t.grad, rdt[sl, :Lr]) <= 1e-5, (precision, rel(t.grad, rdt[sl, :Lr]))
    assert abs(s.grad.item() - rds.item()) <= 1e-5 * abs(rds.item()) + 1e-7, (precision, s.grad.item(), rds.item())

    # (2) whole model step through the public API
    inp = case_inputs(1234, B, E, "spatial")
    x = torch.from_numpy(inp["f"]).to(dev)
    ids, lens = tokens(1234)
    model_1 = build(None, inp, precision)
    model_s = build(G, inp, precision)
    out_1 = model_1.calculate_contrastive_loss(x, ids, lens)
    out_1[0].backward()
    out_s = model_s.calculate_contrastive_loss(x[sl], ids[sl, :Lr], lens[sl])
    out_s[0].backward()
    m.sharding.allreduce_gradients(model_s.parameters(), G)
    l1, ls = out_1[0].item(), out_s[0].item()
    assert abs(l1 - ls) <= 2e-6 * abs(l1), (precision, l1, ls)
    for k in (3, 4):                  # entropies (the accuracies may move by 1/B where the head rounds differently)
        assert abs(out_1[k].item() - out_s[k].item()) <= 1e-5 * abs(out_1[k].item()), (precision, k)
    for (n, p1), (_, ps) in zip(model_1.named_parameters(), model_s.named_parameters()):
        if p1.grad is not None:
            assert rel(ps.grad, p1.grad) <= 5e-3, (precision, n, rel(ps.grad, p1.grad))
    # logits: this rank's [b,b] block of the global matrix
    lpi, lpt = out_s[5], out_s[6]
    ref = out_1[5][sl, sl]
    assert lpi.shape == (b, b) and torch.equal(lpt, lpi.t())
    assert float((lpi - ref).abs().max()) <= 1e-3 * float(ref.abs().max()), precision
    assert out_s[7].shape == (b, E, 7, 7)

# (3) a rank count that differs between ranks: every rank raises the same ValueError (no collective left hanging)
if world > 1:
    nb = b - 1 if rank == 0 else b
    try:
        m.ops.spatial_max_infonce(img[:nb], tok[:nb], lens[:nb], ids[:nb], S, G)
        raise AssertionError("unequal pair counts were not rejected")
    except ValueError as exc:
        assert "same number of pairs" in str(exc)

torch.cuda.synchronize(); dist.barrier()
if rank == 0:
    print("SHARDED_SPATIAL_OK world=%d B=%d L=%s" % (world, B, Ls))
dist.destroy_process_group()
