"""Per-rank compute of the sharded spatial "max" InfoNCE (ops.spatial_max_infonce) next to the single-GPU step.

    python tools/time_sharded_spatial_max.py [--out FILE] [--reps N]

One GPU: an emulated rank (rank 0: row block [b,N] + column block [N,b], the arithmetic a real rank runs after its
gathers) at BASELINE config 4 (B = 1024 pairs, 7x7 map, L = 25, E = 512) for world 1, 2, 4, 8 in both precision
modes, forward and backward timed separately with CUDA events, and the single-GPU step (spatial_max_similarity +
infonce_from_match, forward and backward) on the same batch; then one rank of B = 8192 at world 8 (b = 1024), a batch
whose one-device backward does not fit.  With two or more GPUs, the real sharded op (gathers included) under torchrun
at every world size that fits.  Inputs are leaf feature tensors (the projection head and text encoder are not
timed); operands are not flushed from L2 between repetitions (the B = 1024 fp32 maps alone are 103 MB).  The card's
name and power limit are read in the same run and written beside the numbers."""
import argparse
import json
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

L, HW, E = 25, 49, 512
S = float(-np.log(0.07))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()


def batch(B, dev, seed=4):
    from oracle import cvcl_oracle as O
    gen = torch.Generator(device=dev).manual_seed(seed)
    img = torch.nn.functional.normalize(torch.randn(B, HW, E, device=dev, generator=gen), dim=-1)
    tok = torch.nn.functional.normalize(torch.randn(B, L, E, device=dev, generator=gen), dim=-1)
    ids, lens = O.synth_tokens(np.random.RandomState(seed), B, L, 2350)
    ids = torch.from_numpy(ids).to(dev); lens = torch.from_numpy(lens).to(dev)
    tok = tok * (torch.arange(L, device=dev)[None, :] < lens[:, None])[..., None]
    return img, tok, lens, ids


def timed(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a = torch.cuda.Event(enable_timing=True); c = torch.cuda.Event(enable_timing=True)
        a.record(); fn(); c.record(); c.synchronize()
        ts.append(a.elapsed_time(c))
    return float(np.median(ts)), float(np.min(ts))


def emulated_rank(m, img, tok, lens, ids, world, split, reps):
    """rank 0 of `world`: forward (both blocks + block InfoNCE) and backward (both spatial_max_bwd) in ms"""
    B = img.shape[0]
    b = B // world
    ops = m.ops
    if split:
        gi, gt = img, tok
    else:
        gi = ops.to_bf16_pair(img.reshape(-1, E), False)[0].view(img.shape)
        gt = ops.to_bf16_pair(tok.reshape(-1, E), False)[0].view(tok.shape)
    fwd = ops._spatial_max_block_fwd(split)
    run = lambda: fwd(gi[:b], gt[:b], lens[:b], ids[:b], gi, gt, lens, ids, S, 0, 1.0 / B)
    f_ms, f_min = timed(run, reps)
    out5, l0, l1, _, _, state = run()
    lse0_all = l0.repeat(world); lse1_all = l1.repeat(world)      # values do not change the work
    bwd = lambda: ops._spatial_max_block_bwd(state, 0, 0.5 / B, l0, lse1_all, lse0_all, l1)
    b_ms, b_min = timed(bwd, reps)
    del state
    torch.cuda.empty_cache()
    return dict(world=world, b=b, B=B, fwd_ms=f_ms, fwd_min_ms=f_min, bwd_ms=b_ms, bwd_min_ms=b_min,
                total_ms=f_ms + b_ms)


def single_gpu(m, img, tok, lens, ids, split, reps):
    ops = m.ops
    iv = img.clone().requires_grad_(True); tv = tok.clone().requires_grad_(True)
    s = torch.tensor(S, device=img.device, requires_grad=True)
    fwd = lambda: ops.infonce_from_match(ops.spatial_max_similarity(iv, tv, lens, ids, split=split), s)[0]
    f_ms, f_min = timed(fwd, reps)

    def step():
        fwd().backward()
    t_ms, t_min = timed(step, reps)
    return dict(B=img.shape[0], fwd_ms=f_ms, fwd_min_ms=f_min, total_ms=t_ms, total_min_ms=t_min,
                bwd_ms=t_ms - f_ms)


def real_worker():
    """torchrun target: rank r runs ops.spatial_max_infonce on its b = B/world pairs, forward + backward"""
    import torch.distributed as dist
    rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); lr = int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", lr); torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    import multimodal_baby_b200 as m
    B = int(os.environ["TSSM_B"]); reps = int(os.environ["TSSM_REPS"])
    img, tok, lens, ids = batch(B, dev)
    b = B // world
    sl = slice(rank * b, (rank + 1) * b)
    res = {}
    for precision in ("split_bf16", "bf16"):
        i = img[sl].clone().requires_grad_(True); t = tok[sl].clone().requires_grad_(True)

        def step():
            out = m.ops.spatial_max_infonce(i, t, lens[sl], ids[sl], S, dist.group.WORLD,
                                            split=precision == "split_bf16")
            out[0].backward()
        dist.barrier()
        res[precision] = timed(step, reps)[0]
    if rank == 0:
        print("TSSM " + json.dumps(dict(world=world, B=B, b=b, step_ms=res)))
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_sharded_spatial_max_b200.json"))
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this tool measures on the GPU"
    import multimodal_baby_b200 as m
    m._cabi.load()
    dev = torch.device("cuda", 0)
    res = dict(card=card(), torch=torch.__version__,
               workload="spatial 7x7, sim=max, L=25, E=512, leaf features (head / text encoder not timed)",
               timing="CUDA events, median (and min) of %d repetitions after 2 warm-up calls; L2 not flushed" % a.reps)
    img, tok, lens, ids = batch(1024, dev)
    res["config4_B1024"] = {}
    for precision in ("split_bf16", "bf16"):
        split = precision == "split_bf16"
        r = dict(single_gpu=single_gpu(m, img, tok, lens, ids, split, a.reps), emulated_rank=[])
        for world in (1, 2, 4, 8):
            r["emulated_rank"].append(emulated_rank(m, img, tok, lens, ids, world, split, a.reps))
        one = r["emulated_rank"][0]["total_ms"]
        for q in r["emulated_rank"]:
            q["vs_world1"] = q["total_ms"] / one
        res["config4_B1024"][precision] = r
        print(precision, json.dumps(r), flush=True)
    del img, tok
    torch.cuda.empty_cache()
    img, tok, lens, ids = batch(8192, dev)
    res["B8192_world8_one_rank"] = {}
    for precision in ("split_bf16", "bf16"):
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        q = emulated_rank(m, img, tok, lens, ids, 8, precision == "split_bf16", max(3, a.reps // 3))
        q["peak_gb_above_inputs"] = (torch.cuda.max_memory_allocated() - base) / 1e9
        q["note"] = "the gathered batch is resident (no other rank's data is touched by rank 0's compute)"
        res["B8192_world8_one_rank"][precision] = q
        print("B8192", precision, json.dumps(q), flush=True)
    del img, tok
    torch.cuda.empty_cache()
    n = torch.cuda.device_count()
    res["real_sharded_step"] = []
    for world in (2, 4, 8):
        if n < world:
            res["real_sharded_step"].append(dict(world=world, result="not measured (%d GPU(s) on the machine)" % n))
            continue
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0)); port = sk.getsockname()[1]
        env = dict(os.environ, TSSM_B="1024", TSSM_REPS=str(a.reps))
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__), "--real"]
        p = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=1800)
        line = [x for x in p.stdout.splitlines() if x.startswith("TSSM ")]
        res["real_sharded_step"].append(json.loads(line[0][5:]) if line else
                                        dict(world=world, result="failed: " + p.stderr[-500:]))
    res["card_after"] = card()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    if "--real" in sys.argv:
        real_worker()
    else:
        main()
