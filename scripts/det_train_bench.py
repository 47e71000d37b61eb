"""Deterministic training mode vs the default backward: fwd+bwd step time of one HGTConv layer (C2 shape, d=256, H=8)
and of a 3-layer c4-style stack, with torch.use_deterministic_algorithms off and on ALTERNATED in the same process.
Medians of CUDA-event-timed steps; per-kernel times from a separate torch.profiler run.  Writes a JSON record (card,
power limit, SM clocks beside the numbers) and a short markdown table to --out.

    python scripts/det_train_bench.py --scale 0.25 --steps 20 --out <directory>
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyhgt_b200 import HGTConv, synth, plan as P  # noqa: E402


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = "nvidia-smi unavailable: %s" % e
    return {"query": q, "value": out, "torch_name": torch.cuda.get_device_name(0)}


def build(layers, g, dev):
    torch.manual_seed(0)
    ms = torch.nn.ModuleList([HGTConv(256, 256, g.num_types, g.num_relations, 8, 0.0, True, False)
                              for _ in range(layers)]).to(dev).train()
    x = torch.randn(g.num_nodes, 256, generator=torch.Generator().manual_seed(0)).to(dev)
    w = torch.randn(g.num_nodes, 256, generator=torch.Generator().manual_seed(1)).to(dev)
    args = (g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev))

    def step():
        h = x
        for m in ms:
            h = m(h, *args)
        (h * w).sum().backward()
        ms.zero_grad(set_to_none=True)
    return step


def timed(step, det):
    torch.use_deterministic_algorithms(det)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    step()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def kernel_table(step, det, top=12):
    from torch.profiler import profile, ProfilerActivity
    torch.use_deterministic_algorithms(det)
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    rows = []
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            rows.append((t / 1e3, e.count, e.key[:90]))
    rows.sort(reverse=True)
    return [{"ms": round(t, 3), "calls": c, "kernel": k} for t, c, k in rows[:top]]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=0.25)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "det_train_bench"),
                    help="directory for det_train_bench.json / .md")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    HGTConv.keep_att = False
    g = synth.make_mag_shaped(a.scale)
    rec = {"card": card(), "graph": {"name": "mag-shaped x%g" % a.scale, "nodes": g.num_nodes, "edges": g.num_edges},
           "steps": a.steps, "workloads": {}}
    old = torch.are_deterministic_algorithms_enabled()
    try:
        for name, layers in (("c2_1layer_fwd_bwd", 1), ("c4_3layer_fwd_bwd", 3)):
            P.clear_plan_cache()
            step = build(layers, g, dev)
            for det in (False, True) * a.warmup:
                timed(step, det)
            t = {False: [], True: []}
            for i in range(a.steps):
                for det in ((False, True) if i % 2 == 0 else (True, False)):
                    t[det].append(timed(step, det))
            w = {"default_ms": statistics.median(t[False]), "deterministic_ms": statistics.median(t[True]),
                 "default_ms_all": [round(v, 3) for v in t[False]],
                 "deterministic_ms_all": [round(v, 3) for v in t[True]]}
            w["ratio"] = w["deterministic_ms"] / w["default_ms"]
            w["kernels_default"] = kernel_table(step, False)
            w["kernels_deterministic"] = kernel_table(step, True)
            rec["workloads"][name] = w
            print("%s: default %.3f ms  deterministic %.3f ms  ratio %.3f" % (name, w["default_ms"],
                                                                              w["deterministic_ms"], w["ratio"]),
                  flush=True)
    finally:
        torch.use_deterministic_algorithms(old)
    rec["card_after"] = card()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "det_train_bench.json"), "w") as f:
        json.dump(rec, f, indent=1)
    with open(os.path.join(a.out, "det_train_bench.md"), "w") as f:
        f.write("# Deterministic vs default backward (%s, %s)\n\n" % (rec["graph"]["name"], rec["card"]["value"]))
        f.write("| workload | default ms | deterministic ms | ratio |\n|---|---|---|---|\n")
        for name, w in rec["workloads"].items():
            f.write("| %s | %.3f | %.3f | %.3f |\n" % (name, w["default_ms"], w["deterministic_ms"], w["ratio"]))
        for name, w in rec["workloads"].items():
            for which in ("default", "deterministic"):
                f.write("\n## %s, %s: top kernels (profiler run)\n\n| ms | calls | kernel |\n|---|---|---|\n"
                        % (name, which))
                for r in w["kernels_" + which]:
                    f.write("| %.3f | %d | `%s` |\n" % (r["ms"], r["calls"], r["kernel"]))
    print(json.dumps({k: {"default_ms": v["default_ms"], "deterministic_ms": v["deterministic_ms"]}
                      for k, v in rec["workloads"].items()}))


if __name__ == "__main__":
    main()
