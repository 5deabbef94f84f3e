"""Time the batched spatial-embedding evaluation (MultiModalLitModel.evaluate_trials, embedding_type="spatial").

    python tools/time_eval_spatial.py --out DIR [--runs 20] [--loop-runs 3]

For sim in {max, mean}, E = 512, 7x7 maps, 4-way trials with labels of 3 tokens (22 distinct labels), at the
Labeled-S scale (2200 trials) and the config-5 scale (25 000 trials), CUDA events around:
  (a)  scoring from head outputs [N, 4, E, 7, 7] (layout copy, per-location normalisation, scores, arg-max);
  (a') the scoring kernels alone on normalised NHWC location rows;
  (b)  scoring from layer4 maps [N, 4, 2048, 7, 7], fp32 1x1-conv head included;
  (c)  the per-trial Lightning validation_step loop on the same 2200 trials (the path this replaces).
Warm-up first, then the median of the timed runs.  Algorithmic bytes / flops come from the shapes.  The inputs of
(a) and (b) exceed the 126 MB L2, so no flush is needed between runs; (a') reads 883 MB / 10 GB of rows.
Writes DIR/eval_spatial.json and prints it."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch                                             # noqa: E402
import multimodal_baby_b200 as cv                        # noqa: E402

HBM_BPS = 7.7e12                                         # HGX B200 data sheet, one GPU
L2_BYTES = 126e6
E, K, HW, N_WAY, C, L = 512, 2048, 49, 4, 22, 3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def timed(fn, runs, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(runs):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return {"median_us": statistics.median(ts), "min_us": min(ts), "max_us": max(ts), "runs": runs}


def build(sim, g):
    args = argparse.Namespace(embedding_type="spatial", embedding_dim=E, normalize_features=True, fix_temperature=True,
                              temperature=0.07, text_encoder="embedding", sim=sim)
    vocab = {"<pad>": 0, "<unk>": 1, "<sos>": 2, "<eos>": 3, **{"w%d" % i: i for i in range(4, 2350)}}
    lit = cv.MultiModalLitModel(cv.VisionEncoder(args, trunk="pooled"), cv.TextEncoder(vocab, K, args), args,
                                vocab=vocab)
    with torch.no_grad():
        conv = lit.model.image_embed.model[-1]
        conv.weight.copy_(torch.randn(E, K, 1, 1, generator=g) / 45); conv.bias.copy_(torch.randn(E, generator=g) / 45)
        tab = torch.randn(2350, E, generator=g); tab[0] = 0
        lit.model.text_embed.embedding.weight.copy_(tab)
    return lit.cuda().eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--loop-runs", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_eval_spatial: no CUDA device (timings are GPU-only)")
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(2024)
    ids = torch.zeros((C, L), dtype=torch.int64)
    ids[:, 0], ids[:, 2] = 2, 3
    ids[:, 1] = torch.arange(C) + 100
    lens = torch.full((C,), L, dtype=torch.int64)
    res = {"card": card(), "shapes": dict(E=E, K=K, HW=HW, n_way=N_WAY, labels=C, label_len=L),
           "l2_flushed": False,
           "l2_note": "inputs of (a), (a') and (b) exceed the 126 MB L2 at both scales; no flush between runs",
           "hbm_bound_bps": HBM_BPS, "results": []}
    for n in (2200, 25000):
        M = n * N_WAY
        gd = torch.Generator(device=dev).manual_seed(n)
        index = torch.randint(0, C, (n,), generator=gd, device=dev, dtype=torch.int32)
        maps = torch.empty((n, N_WAY, K, 7, 7), device=dev).normal_(generator=gd).relu_()
        for sim in ("max", "mean"):
            lit = build(sim, g)
            w, b = lit.model._head()
            d_ids, d_lens = ids.to(dev), lens.to(dev)
            with torch.no_grad():
                heads = cv.ops.conv1x1_f32(maps.view(M, K, 7, 7), w, b).view(n, N_WAY, 7, 7, E).permute(0, 1, 4, 2, 3).contiguous()
                rows = cv.ops.normalize_rows_f32(heads.permute(0, 1, 3, 4, 2).reshape(M * HW, E)).view(M, HW, E)
                txt = lit._spatial_text(d_ids, d_lens, HW)
            s = float(lit.model.logit_neg_log_temperature)
            if sim == "max":
                kernels = lambda: cv.ops._spatial_max_scores(rows, txt, d_lens, index, N_WAY, s)     # noqa: E731
                flops_score = 2.0 * M * HW * L * E
            else:
                kernels = lambda: cv.ops.eval_nway(cv.ops.spatial_pool(rows), txt, index, N_WAY, False, s)  # noqa: E731
                flops_score = 1.0 * M * HW * E + 2.0 * M * E
            fa = lambda: lit.evaluate_trials(heads, d_ids, d_lens, index, from_trunk_boundary=False)  # noqa: E731
            fb = lambda: lit.evaluate_trials(maps, d_ids, d_lens, index)                             # noqa: E731
            with torch.no_grad():
                pa, la = fa()
                pb, lb = fb()
            bytes_heads = 4.0 * M * HW * E
            bytes_maps = 4.0 * M * HW * K + 4.0 * E * K
            flops_head = 2.0 * M * HW * E * K
            entry = {"sim": sim, "trials": n, "frames": M}
            with torch.no_grad():
                ta, tk, tb = timed(fa, a.runs), timed(kernels, a.runs), timed(fb, a.runs)
            for name, tm, nbytes, flops in (("a_from_head_outputs", ta, bytes_heads, flops_score),
                                            ("a_scoring_kernels_only", tk, bytes_heads, flops_score),
                                            ("b_from_layer4_maps", tb, bytes_maps, flops_head + flops_score)):
                sec = tm["median_us"] * 1e-6
                entry[name] = dict(tm, algorithmic_bytes=nbytes, algorithmic_flops=flops,
                                   achieved_GBps=nbytes / sec / 1e9, achieved_TFLOPs=flops / sec / 1e12,
                                   hbm_bound_fraction=nbytes / HBM_BPS / sec)
            entry["pred_a_equals_b"] = bool(torch.equal(pa, pb))
            entry["max_abs_logit_a_minus_b"] = float((la - lb).abs().max())
            entry["accuracy_b"] = float((pb == 0).float().mean())
            if n == 2200:
                lit.log = lambda *x, **k: None
                host_maps = [maps[i:i + 1] for i in range(n)]
                host_index = index.tolist()

                def loop():
                    acc = 0
                    for i in range(n):
                        r = host_index[i]
                        acc += lit.validation_step((host_maps[i], d_ids[r:r + 1], d_lens[r:r + 1], [["c%d" % r]]), i, 1)["accuracy"]
                    return acc
                with torch.no_grad():
                    loop_acc = loop()
                    tc = timed(loop, a.loop_runs, warmup=1)
                entry["c_per_trial_validation_step_loop"] = tc
                entry["c_accuracy"] = loop_acc / n
                entry["speedup_c_over_b"] = tc["median_us"] / entry["b_from_layer4_maps"]["median_us"]
            res["results"].append(entry)
            print(json.dumps(entry), flush=True)
            del heads, rows, lit
            torch.cuda.empty_cache()
        del maps
        torch.cuda.empty_cache()
    with open(os.path.join(a.out, "eval_spatial.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
