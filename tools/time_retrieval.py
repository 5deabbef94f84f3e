"""Time cross-modal retrieval (ops.retrieval_f32, the body of MultiModalLitModel.evaluate_retrieval).

    python tools/time_retrieval.py --out DIR [--runs 5]

Cases (E = 512, pair mode, k = 10, R@1/5/10, the default 1 GiB score blocks), from features / head outputs:
  flat   25 000 frames x 25 000 texts (the config-5 scale);
  max    2200 x 2200, 7x7 maps, labels of 3 tokens (the Labeled-S scale);
  mean   the same.
For each case, CUDA events around
  (w) the whole call, both directions: scoring, selection, metrics and the one read-back;
  (s) the scoring alone, both directions, on the same row blocks (normalisation / pooling included);
  (k) the selection kernel alone on one full score block (cvcl_rank_topk_f32).
Warm-up first, then the median of the timed runs.  Achieved fp32 FLOP/s of (s) from the shapes; bytes/s of (k) count
one read of the block and are set against 7.7 TB/s (HGX B200 data sheet, one GPU).  The flat score blocks (1 GiB) exceed
the 126 MB L2; the 2200 x 2200 blocks (19 MB) do not, so (k) reads them from L2 there.  The card's name and power limit
are read in the same run.  Writes DIR/retrieval.json and prints it."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch                                             # noqa: E402
import multimodal_baby_b200 as cv                        # noqa: E402

HBM_BPS = 7.7e12
E, HW, L, K_TOP = 512, 49, 3, 10
S = -math.log(0.07)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def timed(fn, runs, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(runs):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return {"median_us": statistics.median(ts), "min_us": min(ts), "max_us": max(ts), "runs": runs}


def scoring_only(sim, img, txt, lens, block_bytes=1 << 30):
    """the score blocks retrieval_f32 builds, without the selection"""
    ops = cv.ops
    n_img, n_txt = img.shape[0], txt.shape[0]
    if sim == "max":
        rows = ops._location_rows(img, True)
        for q0, q1 in ops._row_blocks(n_img, max(1, block_bytes // (4 * n_txt))):
            ops._spatial_max_scores(rows[q0:q1], txt, lens, None, 0, S)
        for q0, q1 in ops._row_blocks(n_txt, max(1, block_bytes // (4 * n_img)), -(-64 // txt.shape[1])):
            ops._spatial_max_scores(rows, txt[q0:q1], lens[q0:q1], None, 0, S).t().contiguous()
        return
    if sim == "flat":
        i, t = ops.normalize_rows_f32(img), ops.normalize_rows_f32(txt)
    else:
        i, t = ops.spatial_pool(ops._location_rows(img, True)), txt
    for a, b in ((i, t), (t, i)):
        for q0, q1 in ops._row_blocks(a.shape[0], max(1, block_bytes // (4 * b.shape[0]))):
            ops.linear_f32(a[q0:q1], b, None)


def selection_only(block, q0):
    M, N = block.shape
    topk = torch.empty((M, K_TOP), dtype=torch.int32, device=block.device)
    val = torch.empty((M, K_TOP), dtype=torch.float32, device=block.device)
    rank = torch.empty((M,), dtype=torch.int32, device=block.device)
    return lambda: cv._cabi.call("cvcl_rank_topk_f32", cv.ops._p(block), N, M, N, q0, None, None, K_TOP,  # noqa: E731
                                 cv.ops._p(topk), cv.ops._p(val), cv.ops._p(rank), cv.ops._stream())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_retrieval: no CUDA device (timings are GPU-only)")
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device("cuda:0")
    res = {"card": card(), "hbm_bound_bps": HBM_BPS, "k": K_TOP, "block_bytes": 1 << 30, "results": []}
    for sim, n in (("flat", 25000), ("max", 2200), ("mean", 2200)):
        g = torch.Generator(device=dev).manual_seed(n)
        if sim == "flat":
            img = torch.randn((n, E), generator=g, device=dev)
            txt = img + 2.0 * torch.randn((n, E), generator=g, device=dev)
            lens = None
            flops = 2.0 * 2 * n * n * E
        else:
            img = torch.randn((n, HW, E), generator=g, device=dev)
            txt = torch.randn((n, L, E) if sim == "max" else (n, E), generator=g, device=dev)
            txt[:, :] += img[:, :L].mean(1, keepdim=True) if sim == "max" else img.mean(1)
            lens = torch.full((n,), L, dtype=torch.int64, device=dev)
            flops = 2.0 * 2 * n * n * (L * HW * E if sim == "max" else E)
        with torch.no_grad():
            whole = lambda: cv.ops.retrieval_f32(img, txt, lens, sim, True, S, k=K_TOP)       # noqa: E731
            out = whole()
            tw = timed(whole, a.runs)
            ts = timed(lambda: scoring_only(sim, img, txt, lens), a.runs)
            q1 = min(n, (1 << 30) // (4 * n))
            if sim == "flat":
                block = cv.ops.linear_f32(cv.ops.normalize_rows_f32(img[:q1]), cv.ops.normalize_rows_f32(txt), None)
            elif sim == "max":
                block = cv.ops._spatial_max_scores(cv.ops._location_rows(img, True), txt, lens, None, 0, S)
            else:
                block = cv.ops.linear_f32(cv.ops.spatial_pool(cv.ops._location_rows(img, True)), txt, None)
            tk = timed(selection_only(block, 0), a.runs * 4)
        block_bytes = 4.0 * block.numel()
        entry = {"sim": sim, "n_img": n, "n_txt": n, "E": E,
                 "w_whole_call": tw, "s_scoring_only": dict(ts, algorithmic_flops=flops,
                                                             achieved_TFLOPs=flops / (ts["median_us"] * 1e-6) / 1e12),
                 "k_selection_kernel_one_block": dict(tk, rows=block.shape[0], keys=block.shape[1],
                                                      bytes_one_read=block_bytes,
                                                      achieved_GBps=block_bytes / (tk["median_us"] * 1e-6) / 1e9,
                                                      hbm_bound_fraction=block_bytes / HBM_BPS / (tk["median_us"] * 1e-6),
                                                      block_in_l2=block_bytes < 126e6),
                 "selection_and_rest_share_of_whole": 1.0 - ts["median_us"] / tw["median_us"],
                 "recall": {d: out[d]["recall"] for d in out},
                 "median_rank": {d: out[d]["median_rank"] for d in out}}
        res["results"].append(entry)
        print(json.dumps(entry), flush=True)
        del img, txt, block, out
        torch.cuda.empty_cache()
    with open(os.path.join(a.out, "retrieval.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
