"""bf16 K'/V' tables (HGTConv.kv_dtype = torch.bfloat16) vs the fp32 layer: fused inference forward of one HGTConv at
C2, C3 and C5-16M (bench.py's generators and shapes), fp32 and bf16 ALTERNATED in one process on the same inputs.

Per config: median of CUDA-event-timed forwards, peak memory of one forward, the edge kernel's and the typed GEMMs'
times from a separate torch.profiler run (algorithmic bytes/s of the edge kernel and its share of the measured HBM peak),
and the relative Frobenius / max-abs error of sampled output rows of the bf16 layer against the fp32 layer.  Writes a
JSON record (card, power limit, clocks beside the numbers) and a markdown table to --out.

    python scripts/bf16_kv_bench.py --steps 30 --out <directory>
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import CONFIGS, make_graph  # noqa: E402
from pyhgt_b200 import HGTConv, plan as P  # noqa: E402

HBM_PEAK_GBS = 6567.7        # measured HBM read bandwidth of the B200 (DESIGN.md section 4)
SAMPLE_ROWS = 65536
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = "nvidia-smi unavailable: %s" % e
    return {"query": q, "value": out, "torch_name": torch.cuda.get_device_name(0)}


def edge_bytes(n_edges, n_dst, d, rte, row_elem_bytes):
    """Algorithmic HBM bytes of one edge-kernel launch: per edge the [K'|V'] row and its index (+ the RTE index), per
    destination Q, the output and row_ptr (bench.py's count, with the row element size as a parameter)."""
    return n_edges * (2 * d * row_elem_bytes + 4 + (4 if rte else 0)) + n_dst * (2 * d * 4 + 4)


def kernel_times(fwd, n_iter=5):
    from torch.profiler import profile, ProfilerActivity
    fwd()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_iter):
            fwd()
        torch.cuda.synchronize()
    rows = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            rows[e.key] = (t / 1e3 / n_iter, e.count // n_iter)
    def total(sub):
        return sum(t for k, (t, _) in rows.items() if sub in k)
    top = sorted(((t, c, k[:100]) for k, (t, c) in rows.items()), reverse=True)[:10]
    return {"edge_ms": total("k_edge_fwd"), "merge_ms": total("k_merge_partials"), "gemm_ms": total("k_typed_linear"),
            "top": [{"ms": round(t, 4), "calls": c, "kernel": k} for t, c, k in top]}


def run_config(name, edges_m, steps, warmup, dev):
    cfg = CONFIGS[name]
    d, H, rte = cfg["d"], cfg["heads"], cfg["rte"]
    P.clear_plan_cache()
    g = make_graph(name, 1.0, edges_m)
    torch.manual_seed(0)
    m = HGTConv(d, d, g.num_types, g.num_relations, H, 0.2, True, rte).to(dev).eval()
    x = torch.randn(g.num_nodes, d, generator=torch.Generator().manual_seed(0)).to(dev)
    args = (g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev), g.edge_time.to(dev) if rte else None)

    def fwd():
        with torch.no_grad():
            return m(x, *args)

    outs, t = {}, {k: [] for k in DTYPES}
    for _ in range(warmup):
        for k, dt in DTYPES.items():
            m.kv_dtype = dt
            outs[k] = fwd()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for i in range(steps):
        for k in (("fp32", "bf16") if i % 2 == 0 else ("bf16", "fp32")):
            m.kv_dtype = DTYPES[k]
            ev[0].record()
            fwd()
            ev[1].record()
            ev[1].synchronize()
            t[k].append(ev[0].elapsed_time(ev[1]))
    rec = {"config": cfg["label"], "nodes": g.num_nodes, "edges": g.num_edges, "d": d, "heads": H, "rte": rte}
    plan = P.get_plan(args[0], args[1], args[2], args[3], g.num_types, g.num_relations)
    rec["kv_table_bytes_fp32"] = (plan.kv_rows + 1) * 2 * d * 4
    for k, dt in DTYPES.items():
        m.kv_dtype = dt
        del outs[k]
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        outs[k] = fwd()
        torch.cuda.synchronize()
        kt = kernel_times(fwd)
        alg = edge_bytes(g.num_edges, g.num_nodes, d, rte, 4 if k == "fp32" else 2)
        rec[k] = {"median_ms": statistics.median(t[k]), "all_ms": [round(v, 4) for v in t[k]],
                  "peak_mem_bytes": torch.cuda.max_memory_allocated() - base, **kt,
                  "edge_alg_bytes": alg}
        if kt["edge_ms"] > 0:
            gbs = alg / (kt["edge_ms"] * 1e-3) / 1e9
            rec[k]["edge_alg_gbs"] = gbs
            rec[k]["edge_share_of_hbm_peak"] = gbs / HBM_PEAK_GBS
    pick = torch.randperm(g.num_nodes, generator=torch.Generator().manual_seed(1))[:SAMPLE_ROWS].to(dev)
    a, b = outs["bf16"].index_select(0, pick).double(), outs["fp32"].index_select(0, pick).double()
    rec["sampled_rows"] = int(pick.numel())
    rec["rel_fro_bf16_vs_fp32"] = float((a - b).norm() / b.norm())
    rec["max_abs_bf16_vs_fp32"] = float((a - b).abs().max())
    rec["bf16_finite"] = bool(torch.isfinite(outs["bf16"]).all())
    rec["speedup"] = rec["fp32"]["median_ms"] / rec["bf16"]["median_ms"]
    rec["edge_speedup"] = rec["fp32"]["edge_ms"] / rec["bf16"]["edge_ms"] if rec["bf16"]["edge_ms"] else None
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2,c3,c5")
    ap.add_argument("--edges-m", type=float, default=16.0, help="C5 edge count in millions (C5-16M)")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "bf16_kv_bench"),
                    help="directory for bf16_kv_bench.json / .md")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    HGTConv.keep_att = False             # as in bench.py: att materialisation is not part of the metric
    rec = {"card": card(), "hbm_peak_gbs": HBM_PEAK_GBS, "steps": a.steps, "configs": {}}
    for name in a.configs.split(","):
        r = run_config(name, a.edges_m, a.steps, a.warmup, dev)
        rec["configs"][name] = r
        print("%s: fp32 %.3f ms  bf16 %.3f ms  speedup %.3f  edge %.3f -> %.3f ms  rel fro %.2e" % (
            name, r["fp32"]["median_ms"], r["bf16"]["median_ms"], r["speedup"], r["fp32"]["edge_ms"],
            r["bf16"]["edge_ms"], r["rel_fro_bf16_vs_fp32"]), flush=True)
    rec["card_after"] = card()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bf16_kv_bench.json"), "w") as f:
        json.dump(rec, f, indent=1)
    with open(os.path.join(a.out, "bf16_kv_bench.md"), "w") as f:
        f.write("# bf16 vs fp32 K'/V' tables, fused inference forward (%s)\n\n" % rec["card"]["value"])
        f.write("| config | E | fp32 ms | bf16 ms | speedup | edge fp32 ms | edge bf16 ms | edge GB/s fp32 / bf16 "
                "(share of %.1f) | GEMM ms fp32 / bf16 | peak MB fp32 / bf16 | rel fro | max abs |\n" % HBM_PEAK_GBS)
        f.write("|---|---|---|---|---|---|---|---|---|---|---|---|\n")
        for name, r in rec["configs"].items():
            f.write("| %s | %d | %.3f | %.3f | %.3f | %.3f | %.3f | %.0f (%.2f) / %.0f (%.2f) | %.3f / %.3f | %.0f / %.0f "
                    "| %.2e | %.2e |\n" % (
                        name, r["edges"], r["fp32"]["median_ms"], r["bf16"]["median_ms"], r["speedup"],
                        r["fp32"]["edge_ms"], r["bf16"]["edge_ms"], r["fp32"].get("edge_alg_gbs", 0),
                        r["fp32"].get("edge_share_of_hbm_peak", 0), r["bf16"].get("edge_alg_gbs", 0),
                        r["bf16"].get("edge_share_of_hbm_peak", 0), r["fp32"]["gemm_ms"], r["bf16"]["gemm_ms"],
                        r["fp32"]["peak_mem_bytes"] / 2 ** 20, r["bf16"]["peak_mem_bytes"] / 2 ** 20,
                        r["rel_fro_bf16_vs_fp32"], r["max_abs_bf16_vs_fp32"]))
        f.write("\nMedians of %d CUDA-event-timed forwards per dtype, fp32 and bf16 alternated; kernel times from a "
                "separate torch.profiler run (mean of 5 forwards).  Card after the run: %s\n"
                % (a.steps, rec["card_after"]["value"]))
    print(json.dumps({k: {"fp32_ms": v["fp32"]["median_ms"], "bf16_ms": v["bf16"]["median_ms"]}
                      for k, v in rec["configs"].items()}))


if __name__ == "__main__":
    main()
