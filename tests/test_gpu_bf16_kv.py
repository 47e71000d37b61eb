"""GPU tests of the bf16 K'/V' inference mode (HGTConv.kv_dtype = torch.bfloat16; run on the B200: ``pytest -m gpu``).

* Kernel contracts: the bf16-output typed GEMM is bit-identical to the fp32 entry point rounded by torch's .bfloat16();
  the bf16-row edge kernel equals the fp32 edge kernel fed the same tables widened with .float(), bit for bit (the
  rows are widened exactly on load and the arithmetic after the load is the same code).
* The layer: against the fp64 emulation of the mode's contract (tests/bf16_kv_oracle.py), with a tolerance at least 4x
  below the emulation's own distance from the fp64 layer, so a pass means "implements this rounding" and not merely
  "some bf16-sized approximation".
* Memory, kernel selection, switching back to fp32, CUDA-graph replay, and the ValueError cases.
"""
import ctypes
import functools

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import hgt_oracle                          # noqa: E402
from pyhgt_b200 import synth                           # noqa: E402
from tests.bf16_kv_oracle import hgt_forward_bf16kv_fp64, rel_fro   # noqa: E402
from tests.conftest import CONV_FIXTURES, load_golden  # noqa: E402

# GPU bf16 layer vs the fp64 emulation, relative Frobenius: at most a quarter of the emulation's distance from fp64 on
# each fixture (measured per fixture below), and never above LAYER_TOL.
LAYER_TOL = 1e-4


def _dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _st():
    return torch.cuda.current_stream().cuda_stream


def _bits(t):
    return t.contiguous().view(torch.int16) if t.dtype == torch.bfloat16 else t.contiguous().view(torch.int32)


# ---- fixtures -------------------------------------------------------------------------------------------------------

def _conv(fx, dev, dtype=torch.bfloat16):
    import pyhgt_b200
    c = fx["cfg"]
    m = pyhgt_b200.HGTConv(c["in_dim"], c["out_dim"], c["num_types"], c["num_relations"], c["n_heads"], 0.2,
                           c["use_norm"], c["use_RTE"])
    m.load_state_dict(fx["state_dict"])
    m.kv_dtype = dtype
    return m.to(dev).eval()


def _run(m, fx, dev):
    with torch.no_grad():
        out = m(fx["node_inp"].to(dev), fx["node_type"].to(dev), fx["edge_index"].to(dev), fx["edge_type"].to(dev),
                fx["edge_time"].to(dev))
    torch.cuda.synchronize()
    return out


def _kw(c):
    return dict(num_types=c["num_types"], num_relations=c["num_relations"], n_heads=c["n_heads"],
                use_norm=c["use_norm"], use_RTE=c["use_RTE"])


@functools.lru_cache(maxsize=None)
def _emulation(name):
    """(bf16 emulation, its relative Frobenius distance from the fp64 layer) of a conv golden."""
    fx = load_golden(name)
    a = (fx["state_dict"], fx["node_inp"], fx["node_type"], fx["edge_index"], fx["edge_type"], fx["edge_time"])
    ref, _ = hgt_oracle.hgt_forward_dense_fp64(*a, **_kw(fx["cfg"]))
    emu, emu_att = hgt_forward_bf16kv_fp64(*a, **_kw(fx["cfg"]))
    return emu, emu_att, rel_fro(emu, ref)


# ---- typed GEMM: bit-identical to the fp32 entry point rounded by .bfloat16() ---------------------------------------

def _gemm_tables(ms, width, dev):
    """One group per entry of `ms` (rows; 0 = empty group), each with two column blocks written interleaved into rows of
    2*width (the [K'|V'] layout); group g reads A rows from a running offset and W rows 2*width*g.."""
    from pyhgt_b200 import plan as P
    groups, cblocks, a0, off = [], [], 0, 0
    for g, m in enumerate(ms):
        groups.append((a0, m, 2 * width * g, 2, len(cblocks), 1))
        cblocks += [(off, 2 * width), (off + width, 2 * width)]
        a0 += m
        off += m * 2 * width
    return P._pack_groups(groups, cblocks, dev), a0, off


def _gemm_pair(K, width, ms, impl, presplit=False, seed=0):
    from pyhgt_b200 import _lib
    dev = _dev()
    gen = torch.Generator().manual_seed(seed)
    tab, rows, n_out = _gemm_tables(ms, width, dev)
    g_dev, g_host, n_g, c_dev = tab
    a = torch.randn(max(rows, 1), K, generator=gen).to(dev)
    w = (torch.randn(2 * width * len(ms), K, generator=gen) / K ** 0.5).to(dev)
    b = torch.randn(2 * width * len(ms), generator=gen).to(dev)
    out32 = torch.full((max(n_out, 1),), float("nan"), device=dev)
    out16 = torch.full((max(n_out, 1),), float("nan"), device=dev).bfloat16()
    sz = ctypes.c_size_t()
    if presplit:
        hi = torch.empty(a.shape, dtype=torch.bfloat16, device=dev)
        lo = torch.empty_like(hi)
        _lib.call("hgt_act_split", a.data_ptr(), K, a.shape[0], K, 0, None, hi.data_ptr(), lo.data_ptr(), _st())
        for fn, out in (("hgt_typed_linear_presplit", out32), ("hgt_typed_linear_presplit_bf16", out16)):
            _lib.call(fn + "_workspace_bytes", g_host.ctypes.data, n_g, K, width, ctypes.byref(sz))
            ws = torch.empty(max(sz.value, 1), dtype=torch.uint8, device=dev)
            _lib.call(fn, hi.data_ptr(), lo.data_ptr(), w.data_ptr(), b.data_ptr(), K, width, g_dev.data_ptr(),
                      g_host.ctypes.data, n_g, c_dev.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(), _st())
    else:
        for fn, out in (("hgt_typed_linear", out32), ("hgt_typed_linear_bf16", out16)):
            _lib.call(fn + "_workspace_bytes", g_host.ctypes.data, n_g, K, width, impl, ctypes.byref(sz))
            ws = torch.empty(max(sz.value, 1), dtype=torch.uint8, device=dev)
            _lib.call(fn, a.data_ptr(), K, w.data_ptr(), b.data_ptr(), K, width, g_dev.data_ptr(), g_host.ctypes.data,
                      n_g, c_dev.data_ptr(), out.data_ptr(), impl, ws.data_ptr(), ws.numel(), _st())
    torch.cuda.synchronize()
    return out32[:n_out], out16[:n_out]


GEMM_CASES = {
    # name: (K, width, rows per group, impl, presplit, kernel that must run)
    "tc3": (128, 256, [700, 300], 2, False, "k_typed_linear_tc3"),        # cb_width % 256 == 0: CTA-pair kernel
    "tc2": (192, 64, [700, 129, 1], 2, False, "k_typed_linear_tc2"),      # single-CTA W-stationary kernel
    "simt": (100, 36, [500, 277], 1, False, "k_typed_linear_simt"),       # fp32 SIMT kernel, odd widths
    "presplit_tc3": (256, 256, [513, 100], 2, True, "k_typed_linear_tc3"),
    "presplit_tc2": (64, 48, [300, 31], 2, True, "k_typed_linear_tc2"),
    "many_groups": (64, 32, [37 + 5 * g for g in range(70)], 2, False, "k_typed_linear_tc2"),   # > 64 groups: chunks
    "many_groups_simt": (40, 24, [11 + g for g in range(70)], 1, False, "k_typed_linear_simt"),
    "empty_groups": (128, 64, [0, 200, 0, 0, 77, 0], 2, False, "k_typed_linear_tc2"),
    "empty_groups_simt": (40, 24, [0, 50, 0], 1, False, "k_typed_linear_simt"),
}


@pytest.mark.parametrize("case", sorted(GEMM_CASES))
def test_bf16_gemm_is_fp32_gemm_rounded(case):
    from torch.profiler import profile, ProfilerActivity
    K, width, ms, impl, presplit, kernel = GEMM_CASES[case]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        o32, o16 = _gemm_pair(K, width, ms, impl, presplit)
    names = [e.key for e in prof.key_averages()]
    for out_t in ("float", "__nv_bfloat16"):
        assert any("%s<%s>" % (kernel, out_t) in n for n in names), (case, kernel, names)
    assert o16.numel() == sum(ms) * 2 * width
    assert torch.equal(_bits(o32.bfloat16()), _bits(o16)), "%s: bf16 output differs from .bfloat16() of fp32" % case


def test_bf16_gemm_one_tile_fallback_for_wide_k():
    """K = 2304: no W-stationary tile fits, the one-tile-per-CTA kernel runs (checked in the profiler) for both outputs."""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        o32, o16 = _gemm_pair(2304, 32, [300, 130], 2)
    names = [e.key for e in prof.key_averages()]
    assert any("k_typed_linear_tc<__nv_bfloat16>" in n for n in names), names
    assert any("k_typed_linear_tc<float>" in n for n in names), names
    assert torch.equal(_bits(o32.bfloat16()), _bits(o16))


# ---- edge kernel: bf16 rows == the same rows widened to fp32 ----------------------------------------------------------

def _graph(n, e, T, R, seed, hub=0, unmatched=False):
    g = synth.make_random(n, e, T, R, seed=seed, sorted_types=True, isolated_frac=0.1, self_loops=10)
    ei, et, tm = g.edge_index, g.edge_type.clone(), g.edge_time
    if hub:
        gen = torch.Generator().manual_seed(seed + 100)
        src = torch.randint(0, n, (hub,), generator=gen)
        ei = torch.cat([ei, torch.stack([src, torch.full_like(src, 3)])], 1)
        et = torch.cat([et, torch.randint(0, R, (hub,), generator=gen)])
        tm = torch.cat([tm, torch.randint(0, 240, (hub,), generator=gen)])
    if unmatched:
        et[::7] = R + 3                                   # relation outside [0,R): zero row, score 0
    return g.node_type, ei, et, tm


def _edge_pair(d, H, rte, variant, n=600, e=5000, T=3, R=3, seed=0, hub=0, unmatched=False, sync_free=False):
    from pyhgt_b200 import _lib, plan as P
    dev = _dev()
    nt, ei, et, tm = _graph(n, e, T, R, seed, hub, unmatched)
    if e == 0:
        ei, et, tm = ei[:, :0], et[:0], tm[:0]
    host_meta = None
    if sync_free:
        counts = torch.bincount(nt, minlength=T).tolist()
        ok = et < R
        pairs = sorted({(int(s), int(r)) for s, r in zip(nt[ei[0][ok]].tolist(), et[ok].tolist())})
        host_meta = {"type_count": counts, "sorted": True, "pairs": pairs}
    plan = P.build_plan(nt.to(dev), ei.to(dev), et.to(dev), tm.to(dev) if rte else None, T, R, host_meta)
    N, E, Pn = plan.n_nodes, plan.n_edges, plan.n_pairs
    gen = torch.Generator().manual_seed(seed + 1)
    q = torch.randn(N, d, generator=gen).to(dev)
    kv = torch.randn(plan.kv_rows + 1, 2 * d, generator=gen).bfloat16().to(dev)
    kv[-1] = 0
    kvr = None
    if rte:
        kvr = (0.5 * torch.randn(Pn * 240 + 1, 2 * d, generator=gen)).bfloat16().to(dev)
        kvr[-1] = 0
    sz = ctypes.c_size_t()
    _lib.call("hgt_edge_workspace_bytes", plan.n_split, d, H, ctypes.byref(sz))
    split = d % 8 == 0

    def run(fn, kv_t, kvr_t):
        agg = torch.full((N, d), float("nan"), device=dev)
        att = torch.full((max(E, 1), H), float("nan"), device=dev)
        hi = torch.zeros((N, d), dtype=torch.bfloat16, device=dev) if split else None
        lo = torch.zeros_like(hi) if split else None
        ws = torch.zeros(sz.value, dtype=torch.uint8, device=dev)
        _lib.call(fn, q.data_ptr(), kv_t.data_ptr(), _lib.ptr(kvr_t), plan.row_ptr.data_ptr(), plan.kv_row.data_ptr(),
                  _lib.ptr(plan.rte_row) if rte else None, plan.csr_eid.data_ptr(), plan.tiles.data_ptr(), plan.n_tiles,
                  plan.n_split, plan.hubs.data_ptr(), plan.n_hubs, N, E, d, H, 1, agg.data_ptr(),
                  att.data_ptr() if E else None, None, _lib.ptr(hi), _lib.ptr(lo), ws.data_ptr(), ws.numel(), variant,
                  _lib.ptr(plan.tile_counts_dev), plan.type_row0_dev.data_ptr(), T, None, _st())
        torch.cuda.synchronize()
        return agg, att[:E], hi, lo

    r16 = run("hgt_edge_forward_bf16kv", kv, kvr)
    r32 = run("hgt_edge_forward", kv.float(), None if kvr is None else kvr.float())
    return plan, r16, r32


def _check_edge(r16, r32, what):
    for name, a, b in zip(("agg", "att", "hi", "lo"), r16, r32):
        if a is None:
            continue
        assert torch.isfinite(a.float()).all(), "%s %s: non-finite" % (what, name)
        if name in ("agg", "att") and a.numel():
            assert rel_fro(a, b) <= 1e-6, "%s %s: rel fro %.3g" % (what, name, rel_fro(a, b))
        assert torch.equal(_bits(a), _bits(b)), "%s %s: not bitwise equal" % (what, name)


@pytest.mark.parametrize("variant", [1, 2])
@pytest.mark.parametrize("rte", [False, True])
@pytest.mark.parametrize("dk,H", [(4, 8), (16, 4), (25, 4), (32, 8), (50, 2), (32, 32), (4, 1)])
def test_bf16_edge_kernel_matches_widened_fp32(dk, H, rte, variant):
    plan, r16, r32 = _edge_pair(dk * H, H, rte, variant, seed=dk + H)
    _check_edge(r16, r32, "d_k=%d H=%d rte=%s variant=%d" % (dk, H, rte, variant))


@pytest.mark.parametrize("variant", [1, 2])
def test_bf16_edge_kernel_split_hubs_and_unmatched_edges(variant):
    plan, r16, r32 = _edge_pair(256, 8, True, variant, hub=5000, unmatched=True, seed=4)
    assert plan.n_split > 0 and plan.n_hubs > 0
    _check_edge(r16, r32, "hubs + unmatched, variant %d" % variant)


@pytest.mark.parametrize("variant", [1, 2])
def test_bf16_edge_kernel_device_tile_counts(variant):
    plan, r16, r32 = _edge_pair(128, 4, True, variant, hub=3000, seed=6, sync_free=True)
    assert plan.tile_counts_dev is not None and plan.n_split > 0
    _check_edge(r16, r32, "sync-free plan, variant %d" % variant)


@pytest.mark.parametrize("variant", [1, 2])
def test_bf16_edge_kernel_without_edges(variant):
    plan, r16, r32 = _edge_pair(64, 4, False, variant, e=0, seed=8)
    assert plan.n_edges == 0
    _check_edge(r16, r32, "E = 0")
    assert torch.all(r16[0] == 0)


# ---- the layer ------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("variant", [1, 2])
@pytest.mark.parametrize("name", CONV_FIXTURES)
def test_bf16_layer_implements_the_rounding(name, variant, fused):
    dev = _dev()
    fx = load_golden(name)
    m = _conv(fx, dev)
    m.edge_variant, m.fused_call = variant, fused
    out = _run(m, fx, dev).cpu()
    emu, emu_att, emu_dist = _emulation(name)
    assert torch.isfinite(out).all()
    tol = min(LAYER_TOL, emu_dist / 4)
    fro = rel_fro(out, emu)
    assert fro <= tol, "%s (variant %d, fused %s): rel fro vs emulation %.3g > %.3g (emulation vs fp64 %.3g)" % (
        name, variant, fused, fro, tol, emu_dist)
    assert rel_fro(m.att.cpu(), emu_att) <= tol


def _gnn_emulation(fx):
    c = fx["cfg"]
    sd = {k: v.double() for k, v in fx["state_dict"].items()}
    x = fx["node_feature"].double()
    nt = fx["node_type"]
    h = torch.zeros(x.shape[0], c["n_hid"], dtype=torch.float64)
    for t in range(c["num_types"]):
        sel = nt == t
        h[sel] = torch.tanh(x[sel] @ sd["adapt_ws.%d.weight" % t].t() + sd["adapt_ws.%d.bias" % t])
    outs = {}
    for rnd in (True, False):
        y = h
        for layer in range(c["n_layers"]):
            pre = "gcs.%d.base_conv." % layer
            params = {k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}
            norm = c["last_norm"] if layer == c["n_layers"] - 1 else c["prev_norm"]
            y, _ = hgt_forward_bf16kv_fp64(params, y, nt, fx["edge_index"], fx["edge_type"], fx["edge_time"],
                                           num_types=c["num_types"], num_relations=c["num_relations"],
                                           n_heads=c["n_heads"], use_norm=norm, use_RTE=c["use_RTE"], round_kv=rnd)
        outs[rnd] = y
    return outs[True], rel_fro(outs[True], outs[False])


def test_bf16_gnn_stack_matches_emulation():
    import pyhgt_b200
    from pyhgt_b200.model import GNN
    dev = _dev()
    fx = load_golden("gnn_2layer")
    c = fx["cfg"]
    m = GNN(c["in_dim"], c["n_hid"], c["num_types"], c["num_relations"], c["n_heads"], c["n_layers"], 0.2, "hgt",
            c["prev_norm"], c["last_norm"], c["use_RTE"])
    m.load_state_dict(fx["state_dict"], strict=True)
    m = pyhgt_b200.set_kv_dtype(m.to(dev).eval(), torch.bfloat16)
    with torch.no_grad():
        out = m(fx["node_feature"].to(dev), fx["node_type"].to(dev), fx["edge_time"].to(dev), fx["edge_index"].to(dev),
                fx["edge_type"].to(dev)).cpu()
    assert torch.isfinite(out).all()
    emu, emu_dist = _gnn_emulation(fx)
    fro = rel_fro(out, emu)
    assert fro <= min(LAYER_TOL, emu_dist / 4), "GNN: rel fro vs emulation %.3g (emulation vs fp64 %.3g)" % (fro, emu_dist)


def test_switching_back_to_fp32_is_bitwise_the_fp32_result():
    dev = _dev()
    for name in ("c1_rte", "mag_mini_dk50"):
        fx = load_golden(name)
        m = _conv(fx, dev, torch.float32)
        for fused in (True, False):
            m.fused_call = fused
            m.kv_dtype = torch.float32
            ref = _run(m, fx, dev).clone()
            m.kv_dtype = torch.bfloat16
            b16 = _run(m, fx, dev).clone()
            m.kv_dtype = torch.float32
            again = _run(m, fx, dev)
            assert not torch.equal(b16, ref)
            assert torch.equal(_bits(again), _bits(ref)), "%s fused=%s: fp32 after bf16 differs" % (name, fused)


def test_mag_shaped_graph_memory_and_kernels():
    """A mag-shaped graph (x0.05): the bf16 layer's peak memory is lower by at least the K'/V' table saving, and the
    profiler shows the bf16 kernels, not the fp32 edge kernel."""
    import pyhgt_b200
    from pyhgt_b200 import plan as P
    from torch.profiler import profile, ProfilerActivity
    dev = _dev()
    g = synth.make_mag_shaped(0.05)
    d, H = 256, 8
    torch.manual_seed(0)
    m = pyhgt_b200.HGTConv(d, d, g.num_types, g.num_relations, H, 0.2, True, False).to(dev).eval()
    m.keep_att = False
    x = torch.randn(g.num_nodes, d, device=dev)
    args = (g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev))
    peaks, outs = {}, {}
    for dt in (torch.float32, torch.bfloat16, torch.float32, torch.bfloat16):
        m.kv_dtype = dt
        with torch.no_grad():
            outs[dt] = m(x, *args)                     # warm: plan and tables cached
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        with torch.no_grad():
            o = m(x, *args)
        torch.cuda.synchronize()
        peaks[dt] = torch.cuda.max_memory_allocated() - base
        del o
    plan = P.get_plan(args[0], args[1], args[2], None, g.num_types, g.num_relations)
    saving = (plan.kv_rows + 1) * 2 * d * 2
    assert peaks[torch.float32] - peaks[torch.bfloat16] >= saving, (peaks, saving)
    assert torch.isfinite(outs[torch.bfloat16]).all()
    assert rel_fro(outs[torch.bfloat16], outs[torch.float32]) < 2e-3
    for fused in (True, False):
        m.fused_call = fused
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            with torch.no_grad():
                m(x, *args)
            torch.cuda.synchronize()
        names = [e.key for e in prof.key_averages()]
        assert any("k_edge_fwd" in n and "__nv_bfloat16" in n for n in names), names
        assert not any("k_edge_fwd" in n and "<float" in n for n in names), names
        assert any("k_typed_linear_tc" in n and "<__nv_bfloat16>" in n for n in names), names
    m.fused_call = True


def test_graphed_replay_in_bf16_is_bitwise_eager():
    import pyhgt_b200
    from pyhgt_b200.model import GNN
    from pyhgt_b200 import graphed
    dev = _dev()
    T, R, F_in, n_hid = 3, 4, 48, 64
    torch.manual_seed(3)
    m = pyhgt_b200.set_kv_dtype(GNN(F_in, n_hid, T, R, 4, 2, 0.2, "hgt", True, False, True).to(dev).eval(),
                                torch.bfloat16)
    batches = [synth.make_random(n, e, T, R, seed=s, sorted_types=True, self_loops=20)
               for n, e, s in ((400, 3000, 1), (310, 2200, 2))]
    counts = [max(int((b.node_type == t).sum()) for b in batches) + 5 for t in range(T)]
    pairs = {(int(b.node_type[s_]), int(r_)) for b in batches for s_, r_ in zip(b.edge_index[0].tolist(), b.edge_type.tolist())}
    sig = graphed.GraphSignature(counts, 3600, pairs, R, F_in, use_time=True)
    fn = lambda x, nt, tm, ei, et: m(x, nt, tm, ei, et)    # noqa: E731
    g = graphed.GraphedForward(fn, sig, dev)
    old_keep, pyhgt_b200.HGTConv.keep_att = pyhgt_b200.HGTConv.keep_att, False
    try:
        _replay_batches(g, fn, batches, F_in)
    finally:
        pyhgt_b200.HGTConv.keep_att = old_keep


def _replay_batches(g, fn, batches, F_in):
    for b in batches:
        x = torch.randn(b.num_nodes, F_in, generator=torch.Generator().manual_seed(7 + b.num_nodes))
        out = g(x, b.node_type, b.edge_time, b.edge_index, b.edge_type)
        torch.cuda.synchronize()
        replayed = g.out.clone()
        with torch.no_grad():
            eager = fn(g.x, g.nt, g.tm, g.ei, g.et)         # the same padded batch, eagerly, on the same plan
        torch.cuda.synchronize()
        assert torch.equal(_bits(replayed), _bits(eager)), "N=%d: replay differs from eager" % b.num_nodes
        assert torch.isfinite(out).all()


def test_value_errors_raise_before_any_launch():
    import pyhgt_b200
    from pyhgt_b200 import _lib, sharded
    dev = _dev()
    fx = load_golden("c1_rte")
    a = (fx["node_inp"].to(dev), fx["node_type"].to(dev), fx["edge_index"].to(dev), fx["edge_type"].to(dev),
         fx["edge_time"].to(dev))
    m = _conv(fx, dev)
    sh = sharded.ShardedGraph.build(fx["node_type"], fx["edge_index"], fx["edge_type"], fx["edge_time"],
                                    fx["cfg"]["num_types"], fx["cfg"]["num_relations"], 0, 1, dev)
    c = fx["cfg"]
    dense = pyhgt_b200.DenseHGTConv(c["in_dim"], c["out_dim"], c["num_types"], c["num_relations"], c["n_heads"],
                                    0.2, True, True).to(dev).eval()
    dense.kv_dtype = torch.bfloat16
    torch.cuda.synchronize()
    n0 = _lib.kernel_launches()
    m.kv_dtype = torch.float16
    with pytest.raises(ValueError, match="kv_dtype"):
        with torch.no_grad():
            m(*a)
    m.kv_dtype = torch.bfloat16
    with pytest.raises(ValueError, match="inference"):
        m(*a)                                                 # grad enabled and parameters require grad
    with pytest.raises(ValueError, match="inference"):
        m(a[0].clone().requires_grad_(True), *a[1:])
    with pytest.raises(ValueError, match="DenseHGTConv"):
        with torch.no_grad():
            dense(*a)
    with pytest.raises(ValueError, match="sharded"):
        with torch.no_grad():
            sh.forward(m, a[0])
    with pytest.raises(ValueError, match="sharded"):
        sh.forward_train(m, a[0])
    torch.cuda.synchronize()
    assert _lib.kernel_launches() == n0


def test_conv_forward_rejects_an_fp32_layout_with_kv_bf16():
    """hgt_conv_forward with kv_bf16 set on an argument block built for fp32 tables returns an error before launching
    anything, instead of writing bf16 rows at fp32 offsets."""
    import pyhgt_b200
    from pyhgt_b200 import _lib
    dev = _dev()
    fx = load_golden("c1_rte")
    m = _conv(fx, dev, torch.float32)
    _run(m, fx, dev)
    a = next(iter(m._args_cache.values()))[0]
    assert a.kv_bf16 == 0
    bad = _lib.ConvArgs.from_buffer_copy(a)
    bad.kv_bf16, bad.n_q_groups = 1, 0
    wsb = ctypes.c_size_t()
    _lib.call("hgt_conv_workspace_bytes", ctypes.byref(bad), ctypes.byref(wsb))
    ws = torch.empty(wsb.value, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    n0 = _lib.kernel_launches()
    with pytest.raises(_lib.HgtError, match="kv_bf16"):
        _lib.call("hgt_conv_forward", ctypes.byref(bad), ws.data_ptr(), ws.numel(), _st())
    assert _lib.kernel_launches() == n0
