"""bench.py — HGTConv forward edges/s on synthetic heterographs shaped like BASELINE.json's configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c5|c4]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--config (default c2 = the configuration BASELINE.json's metric is quoted on):
  c2  ogbn-mag-shaped, 4 types / 4 relations, N=1.94 M, E=21.1 M, d=256, H=8, no RTE
  c3  OAG-CS-shaped sampled subgraph, 6 types / 10 relations, N=200 k, E=5 M, d=400 (d_k=50), H=8, RTE
  c5  power-law heterograph, 4 types / 8 relations, E = --edges-m million (default 64), N=E/10, d=128, H=8
  c4  the c2 graph through a 3-layer HGTConv stack, forward + backward (training step without the optimiser),
      unit "edge-layers/s"; sharded runs use ShardedGraph.forward_train + gradient all-reduce

One "step" = one HGTConv.forward (pyHGT/conv.py:56) over the whole synthetic graph (c4: fwd+bwd of the stack).
  value     edges/s with every input already resident in HBM and the per-graph plan (CSR) built before the
            timed region; EVERY step is timed by its own CUDA-event pair, per-step max over ranks, and the
            MEDIAN step is reported (SURVEY.md §8d); mean / min / max and the list are in `step_ms`.
  e2e       the same metric through the public module call with HOST (pinned) buffers: every step copies
            node features + node_type + edge_index + edge_type host->device, rebuilds the plan, runs the
            forward and copies the [N,d] result device->host (N > 1: every rank does exactly that for its shard).
  roofline  fused edge kernel (csrc/edge.cu): algorithmic bytes per launch / CUDA-event duration of that
            launch on its own stream, against the measured HBM peak in MEASURED_PEAKS.json.
  cpu_baseline  the CPU oracle port (oracle/hgt_oracle.py: the reference's per-triple algorithm) timed on the
            host cores on a bounded sample (the same generator at a reduced scale), edges/s.
N > 1: destination-node sharding (pyhgt_b200/sharded.py), one halo exchange of source rows per layer; the total
graph is fixed, so scaling is "strong".  Every N > 1 line carries `parity_max_abs_diff`: sampled destination rows
of every rank recomputed by the single-GPU path on their 1-hop induced subgraph, max over ranks, and
`halo_modes_max_abs_diff` (NCCL all-to-all vs NVLink pull kernel).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "HGTConv fwd edges/sec"
UNIT = "edges/s"
FALLBACK_HBM_GBS = 6650.0        # /opt/skills/guides/B200_PROFILING.md fallback

# name -> model shape + CPU-sample scale (the reference materialises ~6 GB per 1 M edges at d=256)
CONFIGS = {
    "c2": dict(d=256, heads=8, rte=False, cpu_scale=0.05, label="c2 ogbn-mag-shaped"),
    "c3": dict(d=400, heads=8, rte=True, cpu_scale=0.1, label="c3 OAG-CS-shaped sampled subgraph"),
    "c5": dict(d=128, heads=8, rte=False, cpu_scale=None, label="c5 power-law heterograph"),
    "c4": dict(d=256, heads=8, rte=False, cpu_scale=0.02, label="c4 ogbn-mag-shaped, 3-layer stack fwd+bwd", layers=3),
}
CPU_SCALE_ENV = os.environ.get("HGT_BENCH_CPU_SCALE")


def make_graph(config, scale=1.0, edges_m=64.0):
    from pyhgt_b200 import synth
    if config in ("c2", "c4"):
        return synth.make_mag_shaped(scale)
    if config == "c3":
        return synth.make_oag_shaped(scale)
    if config == "c5":
        return synth.make_powerlaw(int(edges_m * 1e6 * scale))
    raise SystemExit("unknown --config %r" % config)


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region.  In-process NVML (nvidia_ml_py) when available:
    nvmlInit happens in start() — long before the timed loop — so no driver-wide initialisation can land inside
    it (round 1: an `nvidia-smi -lms` child started next to the warm-up stalled the N=1 run on the 8-GPU box).
    Falls back to the nvidia-smi recipe line, started early and waited for."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, gpu_index=0, pci_bus_id=None):
        self.idx, self.bus = gpu_index, pci_bus_id
        self.samples = []            # (t, sm_mhz, max_mhz, reasons tuple)
        self.mode = None
        self._stop = threading.Event()
        self.t0 = self.t1 = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.bus:
                try:
                    h = pynvml.nvmlDeviceGetHandleByPciBusId(self.bus.encode() if isinstance(self.bus, str) else self.bus)
                except Exception:
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def pump():
                while not self._stop.is_set():
                    try:
                        sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        bits = int(get_reasons(h))
                        self.samples.append((time.perf_counter(), sm, mx,
                                             tuple(n for n, b in self.BITS if bits & b)))
                    except Exception:
                        pass
                    self._stop.wait(0.05)
            self.mode = "nvml"
            self.thread = threading.Thread(target=pump, daemon=True)
            self.thread.start()
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)

            def pump_smi():
                for line in self.proc.stdout:
                    f = [x.strip() for x in line.split(",")]
                    if len(f) < 7:
                        continue
                    try:
                        sm, mx = float(f[0]), float(f[1])
                    except ValueError:
                        continue
                    rs = tuple(n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                                  "sw_power_cap"), f[3:7]) if v.lower().startswith("active"))
                    self.samples.append((time.perf_counter(), sm, mx, rs))
            self.mode = "nvidia-smi"
            self.thread = threading.Thread(target=pump_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.mode = None

    def wait_first(self, timeout=15.0):
        t_end = time.perf_counter() + timeout
        while self.mode and not self.samples and time.perf_counter() < t_end:
            time.sleep(0.05)

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        self._stop.set()
        if self.mode == "nvidia-smi":
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        inside = [s for s in self.samples if self.t0 is not None and self.t0 <= s[0] <= (self.t1 or 1e30)]
        use = inside if inside else self.samples
        sm = sorted(s[1] for s in use)
        reasons = sorted({r for s in use for r in s[3]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max((s[2] for s in use), default=None),
                "reasons": reasons, "samples": len(use), "source": self.mode,
                "window": "timed region" if inside else "whole run (timed region shorter than the sampling period)"}


def edge_algorithmic_bytes(n_edges, n_dst, d, use_rte=False):
    """SURVEY.md §8(d): E*(2*d*4 [K'|V' row] + 4 [kv_row]) + N_dst*(d*4 [Q] + d*4 [agg] + 4 [row_ptr])."""
    per_edge = 2 * d * 4 + 4 + (4 if use_rte else 0)
    return n_edges * per_edge + n_dst * (2 * d * 4 + 4)


DUMP_MAX_BYTES = 64 * 2 ** 20
DUMP_SAMPLE_ROWS = 16384


def dump_rows(n_rows, row_bytes, budget):
    """Row ids --dump-outputs writes of an [n_rows, d] output: all of them when they fit `budget` bytes, else a fixed
    seeded sample of DUMP_SAMPLE_ROWS rows in ascending order (the same rows in every run with the same arguments)."""
    import torch
    if n_rows * row_bytes <= budget:
        return torch.arange(n_rows)
    pick = torch.randperm(n_rows, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE_ROWS]
    return pick.sort().values


def gather_rows(out, rows, n_rows, row_global, world):
    """Rows `rows` of an [n_rows, d] output, on the host.  Sharded runs: `out` holds this rank's rows, global ids
    `row_global`; each sampled row is filled in by its owner and summed over ranks (every other rank adds zeros)."""
    import torch
    if world == 1:
        return out.index_select(0, rows.to(out.device)).cpu()
    import torch.distributed as dist
    pos = torch.full((n_rows,), -1, dtype=torch.int64)
    pos[row_global.cpu()] = torch.arange(row_global.numel())
    local = pos[rows]
    mine = local >= 0
    buf = torch.zeros((rows.numel(), out.shape[1]), dtype=out.dtype, device=out.device)
    buf[mine.to(out.device)] = out.index_select(0, local[mine].to(out.device))
    dist.all_reduce(buf)
    return buf.cpu()


def write_outputs(path, arrays):
    """--dump-outputs: every array as <path>/<name>.npy (float32 values, float64 row ids)."""
    import numpy as np
    total = sum(a.numel() * a.element_size() for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, "dump of %d bytes exceeds %d" % (total, DUMP_MAX_BYTES)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a.numpy())


def _median(v):
    s = sorted(v)
    n = len(s)
    return 0.0 if n == 0 else (s[n // 2] if n % 2 else 0.5 * (s[n // 2 - 1] + s[n // 2]))


def bind_to_local_numa(dev_index):
    """Pin this process (and therefore its pinned host buffers, first-touch) to the CPUs next to its GPU."""
    try:
        import torch
        p = torch.cuda.get_device_properties(dev_index)
        bus = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bus) as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "cpus %s" % spec
    except Exception as exc:                       # noqa: BLE001 — best effort, reported in the line
        return "unbound (%s)" % type(exc).__name__
    return "unbound"


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (the reference's algorithm) on the host cores
# ------------------------------------------------------------------------------------------------------------------
def run_cpu_port(config, steps, warmup, edges_m=64.0):
    """Time the CPU oracle port on a bounded sample of `config`; returns (units/s, info, ms per step, graph)."""
    import torch
    from oracle import hgt_oracle
    cfg = CONFIGS[config]
    d, H, rte = cfg["d"], cfg["heads"], cfg["rte"]
    layers = cfg.get("layers", 1)
    train = config == "c4"
    cores = os.cpu_count() or 1
    if config == "c5":
        full_edges = edges_m * 1e6
        scale = 1.0e6 / full_edges                      # 1 M-edge member of the sweep
    else:
        scale = cfg["cpu_scale"]
    if CPU_SCALE_ENV:
        scale = float(CPU_SCALE_ENV)
    probe_scale = min(scale, 0.2 * scale if config != "c2" else 0.01)

    def forward_stack(params_l, x, g):
        kw = dict(num_types=g.num_types, num_relations=g.num_relations, n_heads=H, use_norm=True, use_RTE=rte)
        h = x
        for p in params_l:
            h, _ = hgt_oracle.hgt_forward_ref_port(p, h, g.node_type, g.edge_index, g.edge_type,
                                                   g.edge_time if rte else None, **kw)
        return h

    def one_step(params_l, x, g):
        if train:
            out = forward_stack(params_l, x, g)
            out.square().sum().backward()
            for p in params_l:
                for v in p.values():
                    v.grad = None
        else:
            with torch.no_grad():
                forward_stack(params_l, x, g)

    def setup(sc):
        g = make_graph(config, sc, edges_m)
        ps = [hgt_oracle.init_params(d, d, g.num_types, g.num_relations, H, use_norm=True, use_RTE=rte, seed=i)
              for i in range(layers)]
        if train:
            for p in ps:
                for v in p.values():
                    v.requires_grad_(True)
        x = torch.randn(g.num_nodes, d, generator=torch.Generator().manual_seed(0))
        return g, ps, x

    # "all the host threads it can use": the reference's small eager ops slow down when oversubscribed, so pick
    # the thread count with the best throughput on a small probe and time the sample with that.
    pg, pps, px = setup(probe_scale)
    best_t, best_dt = cores, float("inf")
    for c in sorted({c for c in (8, 16, 32, 64, cores) if c <= cores}):
        torch.set_num_threads(c)
        dts = []
        for _ in range(2):
            t0 = time.perf_counter()
            one_step(pps, px, pg)
            dts.append(time.perf_counter() - t0)
        if min(dts) < best_dt:
            best_t, best_dt = c, min(dts)
    torch.set_num_threads(best_t)
    # bound the sample to ~5 s per step (about 15-25 s of CPU work in total): units/s is ~scale-invariant
    probe_eps = pg.num_edges / best_dt
    full = 5_000_000 if config == "c3" else (edges_m * 1e6 if config == "c5" else 21_111_007)
    scale = max(probe_scale, min(scale, 5.0 * probe_eps / full))
    g, ps, x = setup(scale)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        one_step(ps, x, g)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    ups = layers * g.num_edges * len(times) / total
    info = {"value": ups, "unit": "edge-layers/s" if train else UNIT, "cores": best_t, "host_cores": cores,
            "kind": "port",
            "sample": "%s x%g (N=%d, E=%d, d=%d, H=%d%s), %d timed %s of oracle/hgt_oracle.py:hgt_forward_ref_port "
                      "(torch %d threads), %.1f s" % (cfg["label"], scale, g.num_nodes, g.num_edges, d, H,
                                                      ", RTE" if rte else "", len(times),
                                                      "fwd+bwd steps of the %d-layer stack" % layers if train
                                                      else "forwards", torch.get_num_threads(), total)}
    return ups, info, total / len(times) * 1e3, g, scale


def main_reference(args, rank, world):
    if rank != 0:
        return
    steps = args.steps
    warmup = 1
    cfg = CONFIGS[args.config]
    ups, info, ms, g, scale = run_cpu_port(args.config, steps, warmup, args.edges_m)
    train = args.config == "c4"
    line = {"impl": "reference", "metric": METRIC if not train else "HGT 3-layer fwd+bwd edge-layers/sec",
            "value": ups, "unit": info["unit"], "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%s (bounded CPU sample x%g: N=%d, E=%d), d=%d, n_heads=%d, %d types / %d relations, "
                                   "use_norm, %s" % (cfg["label"], scale, g.num_nodes, g.num_edges, cfg["d"],
                                                     cfg["heads"], g.num_types, g.num_relations,
                                                     "RTE" if cfg["rte"] else "no RTE")},
            "cpu_baseline": info,
            "e2e": {"value": ups, "unit": info["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
def sampled_rows_parity(conv, g, x_host, out_rows, row_global, dev, rte, n_sample=2048, seed=11):
    """max |sharded - single-GPU| over sampled destination rows.  `out_rows[i]` is this rank's output for global node
    `row_global[i]`.  The sampled destinations' 1-hop induced subgraph (their in-edges and those edges' sources) is run
    through the ordinary single-GPU module: a destination's row depends on nothing else (tests/test_gpu_parity.py)."""
    import torch
    gen = torch.Generator().manual_seed(seed)
    n = row_global.numel()
    pick = torch.randperm(n, generator=gen)[:min(n_sample, n)]
    sample = row_global[pick]
    N = g.num_nodes
    sel = torch.zeros(N, dtype=torch.bool)
    sel[sample] = True
    e_sel = sel[g.edge_index[1]].nonzero(as_tuple=True)[0]
    nodes = torch.unique(torch.cat([sample, g.edge_index[0, e_sel]]))
    local = torch.full((N,), -1, dtype=torch.int64)
    local[nodes] = torch.arange(nodes.numel())
    sub_ei = torch.stack([local[g.edge_index[0, e_sel]], local[g.edge_index[1, e_sel]]]).to(dev)
    with torch.no_grad():
        ref = conv(x_host[nodes].to(dev), g.node_type[nodes].to(dev), sub_ei, g.edge_type[e_sel].to(dev),
                   g.edge_time[e_sel].to(dev) if rte else None)
    diff = (out_rows[pick.to(dev)] - ref[local[sample].to(dev)]).abs().max()
    return diff, int(sample.numel())


def main_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from pyhgt_b200 import HGTConv, _lib
    from pyhgt_b200 import plan as hplan

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    affinity0 = os.sched_getaffinity(0)
    numa = None
    sampler = None
    if rank == 0:
        p = torch.cuda.get_device_properties(local_rank)
        bus = None
        try:
            bus = "%08x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        except Exception:
            pass
        sampler = ClockSampler(local_rank, bus)
        sampler.start()                    # NVML / nvidia-smi start-up happens during graph generation, not the loop
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.config == "c4":
        return main_train(args, rank, local_rank, world, dev, sampler, numa, affinity0)
    cfg = CONFIGS[args.config]
    D, HEADS, RTE = cfg["d"], cfg["heads"], cfg["rte"]
    g = make_graph(args.config, args.scale, args.edges_m)
    E, N = g.num_edges, g.num_nodes
    TYPES, RELS = g.num_types, g.num_relations
    torch.manual_seed(0)
    conv = HGTConv(D, D, TYPES, RELS, HEADS, 0.2, True, RTE).to(dev).eval()
    HGTConv.keep_att = False        # att [E,H] materialisation is opt-in (SURVEY §8b); not part of the metric
    gen = torch.Generator().manual_seed(0)
    x_host = torch.randn(N, D, generator=gen)
    hbm_peak, peak_src = _peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    halo_diff = parity = parity_rows = None
    halo_info = None
    if world == 1:
        x = x_host.to(dev)
        nt, ei, et = g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev)
        tm = g.edge_time.to(dev) if RTE else None

        def step():
            return conv(x, nt, ei, et, tm)
        n_dst_local, e_local = N, E
    else:
        from pyhgt_b200 import sharded
        torch.zeros(1, device=dev)
        torch.cuda.synchronize()                      # context / allocator start-up is not part of the partition time
        t0 = time.perf_counter()
        shard = sharded.ShardedGraph.build(g.node_type, g.edge_index, g.edge_type, g.edge_time if RTE else None, TYPES,
                                           RELS, rank, world, dev, halo_mode=args.halo)
        torch.cuda.synchronize()
        build_s = time.perf_counter() - t0
        # the layer input lives in the rank's NVLink-mapped publish area (where a previous layer's epilogue would have
        # written it): no publish copy inside the step
        x_own = shard.input_buffer(D, 0)
        x_own.copy_(x_host[shard.owned_global].to(dev))

        def step():
            return shard.forward(conv, x_own)
        n_dst_local, e_local = shard.n_owned, shard.n_local_edges
        with torch.no_grad():
            o_ship = step().clone()
            mode = shard.halo_mode                                  # resolved by the first exchange (collectively)
            # (1) both halo exchanges give the same rows
            shard.halo_mode = "nccl"
            o1 = shard.forward(conv, x_own).clone()
            dmax = (o1 - o_ship).abs().max().reshape(1)
            shard.halo_mode = mode
            dist.all_reduce(dmax, op=dist.ReduceOp.MAX)
            halo_diff = dmax.item()
            del o1
            # (2) sharded == single GPU on sampled destination rows of EVERY rank
            pd, nrows = sampled_rows_parity(conv, g, x_host, o_ship, shard.owned_global, dev, RTE)
            pd = pd.reshape(1)
            dist.all_reduce(pd, op=dist.ReduceOp.MAX)
            parity, parity_rows = pd.item(), nrows * world
            del o_ship
        hplan.clear_plan_cache()
        halo_info = shard.halo_stats(D) if hasattr(shard, "halo_stats") else None

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            out = step()
        barrier()
        if sampler is not None:
            sampler.wait_first()
        HGTConv.event_sink = []
        launches0 = _lib.kernel_launches()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        barrier()
        if sampler is not None:
            sampler.mark_begin()
        evs[0].record()
        for i in range(args.steps):
            out = step()
            evs[i + 1].record()
        barrier()
        if sampler is not None:
            sampler.mark_end()
        launches = _lib.kernel_launches() - launches0
        if args.dump_outputs:                                         # `out` is the last timed step's result
            rows = dump_rows(N, D * 4 + 8, DUMP_MAX_BYTES)
            sample = gather_rows(out, rows, N, None if world == 1 else shard.owned_global, world)
            if rank == 0:
                write_outputs(args.dump_outputs, {"out": sample, "out_rows": rows.double()})
        per_step = torch.tensor([evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)], device=dev,
                                dtype=torch.float64)
        if world > 1:
            dist.all_reduce(per_step, op=dist.ReduceOp.MAX)          # a step ends when its slowest rank ends
        per_step = per_step.tolist()
        ms_step = _median(per_step)
        edge_ms = [a.elapsed_time(b) for (n, a, b) in HGTConv.event_sink if n == "edge"]
        lin_ms = [a.elapsed_time(b) for (n, a, b) in HGTConv.event_sink if n in ("proj_linear", "upd_linear")]
        stage_lists = {}
        for (n, a, b) in HGTConv.event_sink:
            stage_lists.setdefault(n, []).append(a.elapsed_time(b))
        stages = {k: _median(v) * (len(v) / args.steps) for k, v in stage_lists.items()}
        HGTConv.event_sink = None
        stages_all = None
        if world > 1:                                   # every rank's stage medians: imbalance shows up as halo wait
            names = sorted(stages)
            mine = torch.tensor([stages[n] for n in names], device=dev, dtype=torch.float64)
            allr = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allr, mine)
            stages_all = {n: [round(float(r[i]), 3) for r in allr] for i, n in enumerate(names)}
        clocks = sampler.stop() if sampler is not None else None
        value = E / (ms_step * 1e-3)

        # ---- roofline of the fused edge kernel (this rank's launches) ----
        edge_med_ms = _median(edge_ms)
        alg = edge_algorithmic_bytes(e_local, n_dst_local, D, RTE)
        achieved = alg / (edge_med_ms * 1e-3) / 1e9 if edge_med_ms > 0 else 0.0
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "edge_traffic.json")) as f:
                tj = json.load(f)
            ent = tj.get("configs", {}).get(args.config)
            if ent and world == 1 and args.scale == 1.0 and (args.config != "c5" or ent.get("edges_m") == args.edges_m):
                traffic, traffic_src = ent["dram_bytes_per_launch"], ent["source"]
        except Exception:
            pass
        # SURVEY.md §8(d): claim min(algorithmic bytes, measured DRAM bytes) / t  (tables that fit L2 make B_alg over-count)
        claim = min(alg, traffic) if traffic else alg
        roofline = {"kernel": "k_edge_fwd_tma (csrc/edge.cu)", "bound": "hbm", "achieved": achieved,
                    "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                    "frac_min_alg_traffic": (claim / (edge_med_ms * 1e-3) / 1e9 / hbm_peak) if edge_med_ms > 0 else None,
                    "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
                    "avg_launch_ms": edge_med_ms, "launch_ms_stat": "median of %d launches" % len(edge_ms),
                    "share_of_step": edge_med_ms / ms_step if ms_step else None}

        # ---- typed linears (tcgen05): FLOPs of ONE fp32-equivalent product; the kernel issues 3 bf16 products ----
        lin_total_ms = sum(lin_ms) / max(args.steps, 1)
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                bf16_peak = float(json.load(f)["bf16_tflops"])
        except Exception:
            bf16_peak = 1590.0
        roofline_linear = None
        if world == 1 and lin_total_ms > 0:
            rows_kv = hplan.get_plan(nt, ei, et, tm, TYPES, RELS).kv_rows     # cached plan of this graph
            flops = 2.0 * D * D * (N + 2 * rows_kv + N)
            roofline_linear = {"kernel": "k_typed_linear_tc* (csrc/linear_tc.cu), projection + a_linear launches",
                               "bound": "tensor", "achieved": 3 * flops / (lin_total_ms * 1e-3) / 1e12,
                               "peak": bf16_peak, "unit": "TFLOP/s (bf16 products issued: 3 per fp32-grade product)",
                               "frac": 3 * flops / (lin_total_ms * 1e-3) / 1e12 / bf16_peak,
                               "fp32_equivalent_tflops": flops / (lin_total_ms * 1e-3) / 1e12,
                               "ms_per_step": lin_total_ms, "includes": "operand hi/lo split kernels"}

        # ---- end to end through the module call with HOST buffers ----
        # Every step copies that step's inputs host->device from pinned memory and its [rows,d] result device->host,
        # all inside the timed region.  The loop is software-pipelined over three streams the way a serving loop
        # would be (H2D of step i+1 and D2H of step i-1 overlap the kernels of step i; PCIe is full duplex); the
        # device input buffers are double-buffered and refilled in place, which invalidates the cached plan, so the
        # CSR plan is rebuilt every step — on one GPU for the whole graph, on N GPUs by every rank for its shard
        # (same work per edge at every N; the host-side partition of the graph into shards is outside, like the
        # graph generation is at N = 1).
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        s_cmp = torch.cuda.current_stream()
        numa = bind_to_local_numa(local_rank)      # the pinned staging buffers are first-touched next to the GPU's PCIe root
        if world == 1:
            host_in = [x_host.pin_memory(), g.node_type.pin_memory(), g.edge_index.pin_memory(), g.edge_type.pin_memory()]
            if RTE:
                host_in.append(g.edge_time.pin_memory())
            rows_out = N
        else:
            host_in = [x_host[shard.owned_global].pin_memory(), shard.node_type.cpu().pin_memory(),
                       shard.edge_index.cpu().pin_memory(), shard.edge_type.cpu().pin_memory()]
            if RTE:
                host_in.append(shard.edge_time.cpu().pin_memory())
            rows_out = shard.n_owned
        dev_in = [[torch.empty_like(t, device=dev) for t in host_in] for _ in range(2)]
        host_out = [torch.empty((rows_out, D), dtype=torch.float32).pin_memory() for _ in range(2)]
        h2d = sum(t.numel() * t.element_size() for t in host_in)
        d2h = rows_out * D * 4
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_cmp = [torch.cuda.Event() for _ in range(2)]
        ev_out = [torch.cuda.Event() for _ in range(2)]

        trace = []                                               # (kind, start_event, end_event) of the timed pipeline
        done = []                                                # completion event of every step's D2H
        CHUNK = 8 * 1024 * 1024                                  # elements; the copy engines serve copies FIFO, so the
                                                                 # GB-sized transfers are cut into pieces to let the plan
                                                                 # build's few-KB read-backs / table uploads slip in between

        def chunked_copy(dst, src):
            df, sf = dst.view(-1), src.view(-1)
            for o0 in range(0, df.numel(), CHUNK):
                df[o0:o0 + CHUNK].copy_(sf[o0:o0 + CHUNK], non_blocking=True)

        def issue_h2d(b):
            with torch.cuda.stream(s_in):
                s_in.wait_event(ev_cmp[b])                       # kernels that read this buffer set have finished
                t0 = torch.cuda.Event(enable_timing=True); t0.record(s_in)
                for dt, ht in zip(dev_in[b], host_in):
                    chunked_copy(dt, ht)
                ev_in[b].record(s_in)
                t1 = torch.cuda.Event(enable_timing=True); t1.record(s_in)
                trace.append(("h2d", t0, t1))

        def run_pipeline(k):
            issue_h2d(0)
            for i in range(k):
                b = i & 1
                if i + 1 < k:
                    issue_h2d((i + 1) & 1)
                s_cmp.wait_event(ev_in[b])
                c0 = torch.cuda.Event(enable_timing=True); c0.record(s_cmp)
                di = dev_in[b]
                if world == 1:
                    o = conv(di[0], di[1], di[2], di[3], di[4] if RTE else None)
                else:
                    o = shard.forward(conv, di[0], graph=(di[1], di[2], di[3], di[4] if RTE else None))
                ev_cmp[b].record(s_cmp)
                c1 = torch.cuda.Event(enable_timing=True); c1.record(s_cmp)
                trace.append(("compute", c0, c1))
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_cmp[b])
                    s_out.wait_event(ev_out[b])                  # the previous D2H into this host buffer is done
                    d0 = torch.cuda.Event(enable_timing=True); d0.record(s_out)
                    chunked_copy(host_out[b], o)
                    o.record_stream(s_out)
                    ev_out[b].record(s_out)
                    d1 = torch.cuda.Event(enable_timing=True); d1.record(s_out)
                    trace.append(("d2h", d0, d1))
                    done.append(d1)
            s_cmp.wait_stream(s_out)
            s_cmp.wait_stream(s_in)

        run_pipeline(2)
        barrier()
        k2 = args.steps
        a, b_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        trace.clear()
        done.clear()
        a.record()
        run_pipeline(k2)
        b_ev.record()
        barrier()
        busy = {}
        for kind, e0, e1 in trace:
            busy[kind] = busy.get(kind, 0.0) + e0.elapsed_time(e1) / k2
        # steady-state interval between consecutive results arriving on the host (median), and the plain mean
        gaps = torch.tensor([done[i].elapsed_time(done[i + 1]) for i in range(len(done) - 1)], device=dev,
                            dtype=torch.float64)
        t2 = torch.tensor([a.elapsed_time(b_ev) / k2], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
            if k2 > 1:
                dist.all_reduce(gaps, op=dist.ReduceOp.MAX)
        e2e_ms = _median(gaps.tolist()) if k2 > 1 else t2.item()     # one step has no interval: its whole time
        h2d_all = torch.tensor([float(h2d), float(d2h)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(h2d_all)
        e2e = {"value": E / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_all[0].item()),
               "d2h_bytes_per_step": int(h2d_all[1].item()), "ms_per_step": e2e_ms,
               "ms_per_step_stat": ("median interval between consecutive results landing in host memory "
                                    "(%d steps, max over ranks)" % k2) if k2 > 1 else
                                   "time of the single step, H2D to D2H (max over ranks)",
               "ms_per_step_mean": t2.item(),
               "stream_busy_ms_per_step_rank0": {k: round(v, 2) for k, v in busy.items()},
               "includes": ("per step%s: H2D of node_inp/node_type/edge_index/edge_type%s from pinned host memory, plan "
                            "(CSR) rebuild, %sforward, D2H of out [rows,d]"
                            % ("" if world == 1 else " and rank (its shard: owned feature rows + local graph)",
                               "/edge_time" if RTE else "", "" if world == 1 else "halo exchange, ") +
                            "; 3-stream software pipeline over %d steps (copies of neighbouring steps overlap compute)"
                            % k2),
               "host_numa": numa}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            os.sched_setaffinity(0, affinity0)       # the CPU arm may use every host core again
        except OSError:
            pass
        _, cpu, _, _, _ = run_cpu_port(args.config, steps=3, warmup=1, edges_m=args.edges_m)
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "%s: %d node types / %d relations, N=%d, E=%d, d=%d, n_heads=%d, "
                                       "use_norm, %s, eval/no_grad%s" % (cfg["label"], TYPES, RELS, N, E, D, HEADS,
                                                                         "RTE" if RTE else "no RTE",
                                                                         "" if args.scale == 1.0 else " (scale %g)" % args.scale),
                           "l2": "inputs exceed L2: node features %.2f GB and [K'|V'] table >> 126 MB; no flush needed"
                                 % (N * D * 4 / 1e9),
                           "plan": "destination-sorted CSR built once before the timed region (value); rebuilt every "
                                   "step in e2e",
                           "parallelism": "single GPU" if world == 1 else
                                          "dst-node sharding x%d, halo source rows per step via %s" % (
                                              world, "one NCCL all_to_all_single" if shard.halo_mode == "nccl"
                                              else ("owner-push kernel over NVLink (experimental)" if shard.halo_mode == "push"
                                                    else "fused NVLink peer-memory pull kernel (torch symmetric memory)")),
                           "linear": "tcgen05 split-bf16 (3 products, fp32 accumulate)", "edge": "TMA bulk-copy ring"},
                "step_ms": {"stat": "median of per-step CUDA-event pairs (per-step max over ranks)",
                            "median": ms_step, "mean": sum(per_step) / len(per_step), "min": min(per_step),
                            "max": max(per_step), "list": [round(v, 3) for v in per_step]},
                "roofline": roofline, "roofline_linear": roofline_linear,
                "stage_ms_rank0": {k: round(v, 3) for k, v in stages.items()}, "stage_ms_all_ranks": stages_all,
                "halo_modes_max_abs_diff": halo_diff, "parity_max_abs_diff": parity,
                "parity": None if parity is None else
                "%d sampled destination rows (all ranks) vs the single-GPU path on their 1-hop induced subgraph"
                % parity_rows,
                "halo": halo_info,
                "shard_build_s_rank0": None if world == 1 else round(build_s, 2),
                "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main_train(args, rank, local_rank, world, dev, sampler, numa, affinity0):
    """BASELINE config 4: c2 graph, 3-layer HGTConv stack (d=256, H=8, use_norm, dropout 0), forward + backward with
    gradients for every parameter (OAG/train_paper_field.py:242-252 without the optimiser step); N > 1: destination
    sharding with the differentiable halo exchange and an all-reduce of the parameter gradients."""
    import torch
    import torch.distributed as dist
    from pyhgt_b200 import HGTConv, _lib
    cfg = CONFIGS["c4"]
    D, HEADS, L = cfg["d"], cfg["heads"], cfg["layers"]
    g = make_graph("c4", args.scale)
    E, N, T, R = g.num_edges, g.num_nodes, g.num_types, g.num_relations
    torch.manual_seed(0)
    layers = torch.nn.ModuleList([HGTConv(D, D, T, R, HEADS, 0.0, True, False) for _ in range(L)]).to(dev).train()
    HGTConv.keep_att = False
    x_host = torch.randn(N, D, generator=torch.Generator().manual_seed(0))
    w_host = torch.randn(N, D, generator=torch.Generator().manual_seed(1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if world == 1:
        x, w = x_host.to(dev), w_host.to(dev)
        nt, ei, et = g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev)

        def step():
            h = x
            for m in layers:
                h = m(h, nt, ei, et)
            (h * w).sum().backward()
            return h
    else:
        from pyhgt_b200 import sharded
        shard = sharded.ShardedGraph.build(g.node_type, g.edge_index, g.edge_type, None, T, R, rank, world, dev,
                                           halo_mode="nccl")
        x, w = x_host[shard.owned_global].to(dev), w_host[shard.owned_global].to(dev)

        def step():
            h = x
            for m in layers:
                h = shard.forward_train(m, h)
            (h * w).sum().backward()
            shard.allreduce_grads(layers)
            return h

    for _ in range(max(args.warmup, 3)):
        step()
        layers.zero_grad(set_to_none=True)
    barrier()
    if sampler is not None:
        sampler.wait_first()
    launches0 = _lib.kernel_launches()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    if sampler is not None:
        sampler.mark_begin()
    evs[0].record()
    for i in range(args.steps):
        layers.zero_grad(set_to_none=True)           # at the start, so the last step's gradients outlive the loop
        h = step()
        evs[i + 1].record()
    barrier()
    if sampler is not None:
        sampler.mark_end()
    launches = _lib.kernel_launches() - launches0
    if args.dump_outputs:                            # the last step's output rows and parameter gradients
        grads = {"grad." + n: p.grad.cpu() for n, p in layers.named_parameters() if p.grad is not None}
        rows = dump_rows(N, D * 4 + 8, DUMP_MAX_BYTES - sum(g.numel() * 4 for g in grads.values()))
        sample = gather_rows(h.detach(), rows, N, None if world == 1 else shard.owned_global, world)
        if rank == 0:
            write_outputs(args.dump_outputs, dict(out=sample, out_rows=rows.double(), **grads))
    per_step = torch.tensor([evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(per_step, op=dist.ReduceOp.MAX)
    per_step = per_step.tolist()
    ms_step = _median(per_step)
    clocks = sampler.stop() if sampler is not None else None
    peak_gb = torch.cuda.max_memory_allocated() / 1e9
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            os.sched_setaffinity(0, affinity0)
        except OSError:
            pass
        _, cpu, _, _, _ = run_cpu_port("c4", steps=2, warmup=1)
    if rank == 0:
        value = L * E / (ms_step * 1e-3)
        line = {"metric": "HGT 3-layer fwd+bwd edge-layers/sec", "value": value, "unit": "edge-layers/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "%s: N=%d, E=%d, d=%d, n_heads=%d, %d layers, use_norm, no RTE, dropout 0, "
                                       "train mode, gradients w.r.t. every parameter%s"
                                       % (cfg["label"], N, E, D, HEADS, L,
                                          "" if args.scale == 1.0 else " (scale %g)" % args.scale),
                           "parallelism": "single GPU" if world == 1 else
                                          "dst-node sharding x%d: differentiable halo exchange (all-to-all forward, reverse "
                                          "all-to-all with add backward), parameter-gradient all-reduce" % world},
                "step_ms": {"stat": "median of per-step CUDA-event pairs (per-step max over ranks)", "median": ms_step,
                            "mean": sum(per_step) / len(per_step), "min": min(per_step), "max": max(per_step),
                            "list": [round(v, 3) for v in per_step]},
                "peak_mem_gb_rank0": round(peak_gb, 2), "cpu_baseline": cpu,
                "e2e": None, "gpu_launches": launches, "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--edges-m", type=float, default=64.0, help="c5: millions of edges (sweep member)")
    ap.add_argument("--scale", type=float, default=1.0, help="graph scale (1.0 = the BASELINE size of --config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--halo", default=None, choices=["nccl", "p2p", "push"],
                    help="multi-GPU halo exchange: one NCCL all_to_all or the fused peer-memory pull kernel (default auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (at most 64 MB: "
                         "a fixed seeded sample of the output rows, ids in out_rows.npy; c4 adds grad.<param>.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm times a smaller CPU sample")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        main_reference(args, rank, world)
        return
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun (python -m torch.distributed.run --nproc-per-node %d bench.py ...)"
                             % (args.gpus, args.gpus))
    main_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
