"""world-2/4 `gloo` tests (CPU) of the sharded spatial "max" InfoNCE orchestration
(sharding.spatial_max_infonce_forward / _backward): gathers, ragged utterance lengths, diagonal offsets and the
reductions, with the block arithmetic injected as an fp64 torch restatement (tests/_sharded_spatial.py; the CUDA
ops replace it on the GPU).  Every rank's result must equal single-process autograd of the oracle on the
concatenated batch."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
S = float(-np.log(0.07))
B, E = 24, 32


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q, sizes):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    sys.path.insert(0, HERE)
    from multimodal_baby_b200 import sharding
    import _sharded_spatial as R
    try:
        img, tok, lens, ids, Ls = R.ragged_batch(5, B, E, world)
        if sizes is not None:                              # unequal pair counts: rank r holds sizes[r] pairs
            lo = sum(sizes[:rank])
            sl = slice(lo, lo + sizes[rank])
        else:
            b = B // world
            sl = slice(rank * b, (rank + 1) * b)
        L = Ls[rank] if sizes is None else tok.shape[1]
        try:
            out5, saved, (a0, a1) = sharding.spatial_max_infonce_forward(
                img[sl].contiguous(), tok[sl, :L].contiguous(), lens[sl].contiguous(), ids[sl, :L].contiguous(),
                S, dist.group.WORLD, R.compute_fwd)
        except ValueError as exc:
            q.put((rank, "ValueError", str(exc)))
            return
        dimg, dtok, ds = sharding.spatial_max_infonce_backward(saved, dist.group.WORLD, R.compute_bwd)
        q.put((rank, out5.numpy(), dimg.numpy(), dtok.numpy(), ds.numpy(), a0.numpy(), a1.numpy()))
    finally:
        dist.barrier()
        dist.destroy_process_group()


def _run(world, sizes=None):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, sizes)) for r in range(world)]
    for p in procs:
        p.start()
    results = sorted([q.get(timeout=180) for _ in range(world)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return results


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_spatial_max_equals_single_process(world):
    results = _run(world)
    sys.path.insert(0, ROOT)
    sys.path.insert(0, HERE)
    from oracle import cvcl_oracle as O
    import _sharded_spatial as R
    img, tok, lens, ids, Ls = R.ragged_batch(5, B, E, world)
    assert len(set(Ls)) == world                                    # every rank holds a different L
    img.requires_grad_(True); tok.requires_grad_(True)
    s = torch.tensor(S, dtype=torch.float64, requires_grad=True)
    match = O.similarity_spatial_max(img.permute(0, 2, 1).reshape(B, E, 7, 7), tok, lens)
    ref = O.infonce(*O.logits_from_match(match, s))
    ref.loss.backward()
    b = B // world
    for rank, out5, dimg, dtok, ds, a0, a1 in results:
        sl = slice(rank * b, (rank + 1) * b)
        assert abs(out5[0] - ref.loss.item()) < 1e-12
        assert abs(out5[1] - ref.image_accuracy.item()) < 1e-7      # reference accuracy is fp32
        assert abs(out5[2] - ref.text_accuracy.item()) < 1e-7
        assert abs(out5[3] - ref.image_entropy.item()) < 1e-12
        assert abs(out5[4] - ref.text_entropy.item()) < 1e-12
        assert np.array_equal(a0, ref.image_pred[sl].numpy().astype(np.int32))
        assert np.array_equal(a1, ref.text_pred[sl].numpy().astype(np.int32))
        np.testing.assert_allclose(dimg, img.grad[sl].numpy(), rtol=0, atol=1e-12)
        # tokens: this rank's own L; positions beyond len carry no gradient (the oracle's zero pad rows tie over the
        # locations, and the embedding's padding row drops what it gets there)
        assert dtok.shape == (b, Ls[rank], E)
        valid = (torch.arange(Ls[rank])[None, :] < lens[sl, None]).numpy()
        np.testing.assert_allclose(dtok[valid], tok.grad[sl, :Ls[rank]].numpy()[valid], rtol=0, atol=1e-12)
        assert not dtok[~valid].any()
        assert abs(ds[0] - s.grad.item()) < 1e-12


def test_sharded_spatial_max_unequal_pairs_raise_on_every_rank():
    results = _run(2, sizes=[10, 14])
    assert [r[1] for r in results] == ["ValueError", "ValueError"]
    assert all("same number of pairs" in r[2] for r in results)
