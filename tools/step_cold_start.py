"""Cold-start cost of the one-kernel flat train step, phase by phase (B = 512, bench.py's shapes and seeds).

bench.py times the step with a 256 MiB `zero_()` between steps, which evicts the kernel's code and inputs from
L2 and leaves the cache full of dirty lines.  This runs the same call (ops.flat_contrastive_step on the library
named by CVCL_B200_LIB, else the in-tree build) in three conditions, taken in turn launch after launch:

    warm         no flush: the previous launch of the step has just run
    write-flush  256 MiB zero_() before the step (bench.py's condition)
    read-flush   a reduction over 256 MiB before the step: evicts as much, but leaves clean lines

and prints, per condition, the median CUDA-event step time and the median of each phase's in-kernel duration
(CTA 0's globaltimer stamps, read as bench.fused_phase_timeline reads them).  Cold minus warm is the cost of
fetching code and inputs again; write-flush minus read-flush is the write-back of the flush's dirty lines.

    CVCL_B200_LIB=<lib> python tools/step_cold_start.py [--launches N] [--out FILE.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402

CONDITIONS = ("warm", "write-flush", "read-flush")


def gpu_info(index=0):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return dict(zip(q.split(","), [c.strip() for c in r.stdout.strip().split(",")]))
    except (OSError, subprocess.SubprocessError) as exc:
        return {"error": str(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=300, help="timed launches per condition (at least 200)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", help="also write the JSON result here")
    a = ap.parse_args()
    if a.launches < 200:
        ap.error("--launches must be at least 200")
    if not torch.cuda.is_available():
        raise SystemExit("step_cold_start.py needs a CUDA device")
    dev = torch.device("cuda:0")
    B = 512
    m, model = bench.build_model(dev, None)
    from multimodal_baby_b200 import _cabi
    lib_path = os.environ.get("CVCL_B200_LIB") or "in-tree build"
    if os.path.isabs(lib_path) and lib_path.startswith(ROOT + os.sep):
        lib_path = os.path.relpath(lib_path, ROOT)
    _cabi.load()
    if not m.ops.fused_supported(B, bench.L, bench.E, bench.K, bench.V):
        raise SystemExit("the one-kernel step does not cover B = %d" % B)
    f, ids, lens = bench.synth_batch(1234, B)
    x = torch.from_numpy(f).to(torch.bfloat16).to(dev)
    ids = torch.from_numpy(ids).to(dev)
    lens = torch.from_numpy(lens).to(dev)
    w, b = model.image_embed.model.fc.weight, model.image_embed.model.fc.bias
    table = model.text_embed.embedding.weight
    m.ops.register_weight_shadow(w, w.detach().to(torch.bfloat16).contiguous())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush.zero_()
    flush_f = flush.view(torch.float32)
    sink = torch.empty((), dtype=torch.float32, device=dev)

    def step():
        return m.ops.flat_contrastive_step(x, ids, lens, w, b, table, bench.S_FIXED, True, True, False)

    def prepare(cond):
        if cond == "write-flush":
            flush.zero_()
        elif cond == "read-flush":
            torch.sum(flush_f, dim=0, out=sink)

    for i in range(a.warmup):
        prepare(CONDITIONS[i % 3]); step()
    torch.cuda.synchronize()
    times = {c: [] for c in CONDITIONS}
    phases = {c: {} for c in CONDITIONS}
    sampler = bench.ClockSampler(0)
    sampler.start()
    for i in range(3 * a.launches):
        cond = CONDITIONS[i % 3]
        prepare(cond)
        # keep the GPU busy while the host enqueues the step (~100 us of spinning, no memory traffic): otherwise the
        # warm condition, which has no flush in front of it, would time the host's launch path instead of the step
        torch.cuda._sleep(200000)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); step(); e1.record(); e1.synchronize()
        times[cond].append(e0.elapsed_time(e1) * 1e3)
        for name, us in (bench.fused_phase_timeline(m, B) or {}).items():
            phases[cond].setdefault(name, []).append(us)
    clocks = sampler.stop()
    res = dict(lib=lib_path, pairs=B, launches_per_condition=a.launches, gpu=gpu_info(), clocks_during_run=clocks,
               conditions={})
    for c in CONDITIONS:
        res["conditions"][c] = dict(step_us_median=round(statistics.median(times[c]), 2),
                                    step_us_min=round(min(times[c]), 2),
                                    phases_us_median={k: round(statistics.median(v), 2) for k, v in phases[c].items()})
    warm = res["conditions"]["warm"]
    for c in ("write-flush", "read-flush"):
        cc = res["conditions"][c]
        cc["minus_warm_us"] = dict(step=round(cc["step_us_median"] - warm["step_us_median"], 2),
                                   **{k: round(v - warm["phases_us_median"].get(k, 0.0), 2)
                                      for k, v in cc["phases_us_median"].items()})
    print("library %s   %s" % (lib_path, res["gpu"]))
    names = list(warm["phases_us_median"])
    print("%-42s" % "median us" + "".join("%14s" % c for c in CONDITIONS) + "%14s%14s" % ("write-warm", "read-warm"))
    for k in ["step (CUDA events)"] + names:
        vals = [res["conditions"][c]["step_us_median"] if k.startswith("step") else
                res["conditions"][c]["phases_us_median"].get(k, float("nan")) for c in CONDITIONS]
        print("%-42s" % k[:42] + "".join("%14.2f" % v for v in vals) + "%14.2f%14.2f" % (vals[1] - vals[0], vals[2] - vals[0]))
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
