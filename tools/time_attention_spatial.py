"""Time the text-to-location attention maps of a spatial-embedding model (ops.spatial_attention_f32,
MultiModalLitModel.attention_maps).

    python tools/time_attention_spatial.py --out DIR [--runs 20]

At the Labeled-S scale (2200 frames: 22 categories x 100) and at 22 000 frames, E = 512, 7x7 maps, every frame
against its category label of 3 tokens, CUDA events around:
  (a)  maps from head outputs [M, 49, E] (per-location normalisation pass + the attention kernel);
  (a') the attention kernel alone on normalised location rows;
  (b)  maps from layer4 maps [M, 2048, 7, 7] through the model (fp32 1x1-conv head, text features, kernel).
Warm-up first, then the median of the timed runs.  The bytes each case must read at least come from the shapes
(the head outputs once: M * 49 * E * 4 B, 220.8 MB at 2200 frames, more than the 126 MB L2, so no flush is
needed); the HBM fraction is that floor at 7.7 TB/s over the measured time.  The card's name and power limit are
read in the same call.  Writes DIR/attention_spatial.json and prints it."""
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
E, K, HW, C, L = 512, 2048, 49, 22, 3


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


def build(g):
    args = argparse.Namespace(embedding_type="spatial", embedding_dim=E, normalize_features=True, fix_temperature=True,
                              temperature=0.07, text_encoder="embedding", sim="max")
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
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_attention_spatial: no CUDA device (timings are GPU-only)")
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(2024)
    lit = build(g)
    m = lit.model
    ids = torch.zeros((C, L), dtype=torch.int64)
    ids[:, 0], ids[:, 2] = 2, 3
    ids[:, 1] = torch.arange(C) + 100
    lens = torch.full((C,), L, dtype=torch.int64)
    d_ids, d_lens = ids.to(dev), lens.to(dev)
    with torch.no_grad():
        tok, _ = cv.ops.text_features_spatial(d_ids, d_lens, m.text_embed.embedding.weight, True)
    res = {"card": card(), "shapes": dict(E=E, K=K, HW=HW, labels=C, label_len=L), "l2_flushed": False,
           "l2_note": "the head outputs (220.8 MB at 2200 frames) and the layer4 maps exceed the 126 MB L2",
           "hbm_bound_bps": HBM_BPS, "results": []}
    for M in (2200, 22000):
        gd = torch.Generator(device=dev).manual_seed(M)
        index = torch.randint(0, C, (M,), generator=gd, device=dev, dtype=torch.int32)
        maps = torch.empty((M, K, 7, 7), device=dev).normal_(generator=gd).relu_()
        w, b = m._head()
        with torch.no_grad():
            heads = cv.ops.conv1x1_f32(maps, w, b).view(M, HW, E)
            rows = cv.ops._location_rows(heads, True)
        fa = lambda: cv.ops.spatial_attention_f32(heads, tok, d_lens, index, True)       # noqa: E731
        fk = lambda: cv.ops.spatial_attention_f32(rows, tok, d_lens, index, False)       # noqa: E731
        fb = lambda: lit.attention_maps(maps, d_ids, d_lens, index)                     # noqa: E731
        with torch.no_grad():
            oa, ok, ob = fa(), fk(), fb()
            ta, tk, tb = timed(fa, a.runs), timed(fk, a.runs), timed(fb, a.runs)
        floor_heads = 4.0 * M * HW * E
        out_bytes = 4.0 * M * (L * HW + HW + L)
        entry = {"frames": M, "floor_bytes_head_outputs": floor_heads, "output_bytes": out_bytes,
                 "floor_us_at_7.7TBps": floor_heads / HBM_BPS * 1e6,
                 "kernel_equals_from_head_outputs": all(torch.equal(x, y) for x, y in zip(oa, ok)),
                 "model_equals_from_head_outputs": bool(torch.equal(ob[1].reshape(M, L, HW), oa[0])
                                                        and torch.equal(ob[0].reshape(M, HW), oa[1])
                                                        and torch.equal(ob[2], oa[2]))}
        for name, tm, nbytes, flops in (
                ("a_from_head_outputs", ta, floor_heads, 2.0 * M * HW * L * E),
                ("a_kernel_only", tk, floor_heads, 2.0 * M * HW * L * E),
                ("b_from_layer4_maps", tb, 4.0 * M * HW * K + 4.0 * E * K, 2.0 * M * HW * E * K + 2.0 * M * HW * L * E)):
            sec = tm["median_us"] * 1e-6
            entry[name] = dict(tm, floor_bytes=nbytes, algorithmic_flops=flops, achieved_GBps=nbytes / sec / 1e9,
                               achieved_TFLOPs=flops / sec / 1e12, hbm_bound_fraction=nbytes / HBM_BPS / sec)
        res["results"].append(entry)
        print(json.dumps(entry), flush=True)
        del maps, heads, rows, oa, ok, ob
        torch.cuda.empty_cache()
    with open(os.path.join(a.out, "attention_spatial.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
