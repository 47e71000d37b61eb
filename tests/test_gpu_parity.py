"""GPU parity tests (run on the B200 box: ``pytest -m gpu``).  The CUDA path (through the C ABI) is compared
with (a) golden outputs of the reference itself (tests/golden, made by oracle/make_golden.py) and (b) the CPU
oracle on seeded graphs.  Tolerance from BASELINE.json north_star: 1e-3 (allclose rtol=atol=1e-3 and relative
Frobenius error <= 1e-3); index handling is bit-exact."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import hgt_oracle          # noqa: E402
from pyhgt_b200 import synth           # noqa: E402
from tests.conftest import load_golden, CONV_FIXTURES  # noqa: E402

RTOL = ATOL = 1e-3


def _dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _close(a, b, what, atol=ATOL):
    a, b = a.float().cpu(), b.float().cpu()
    err = (a - b).abs().max().item() if a.numel() else 0.0
    fro = ((a - b).norm() / b.norm().clamp_min(1e-30)).item() if a.numel() else 0.0
    assert torch.allclose(a, b, rtol=RTOL, atol=atol), "%s: max abs err %.3g (rel fro %.3g)" % (what, err, fro)
    assert fro <= 1e-3, "%s: relative Frobenius error %.3g" % (what, fro)


def _module_from_fixture(fx, dev):
    import pyhgt_b200
    c = fx["cfg"]
    m = pyhgt_b200.HGTConv(c["in_dim"], c["out_dim"], c["num_types"], c["num_relations"], c["n_heads"], 0.2,
                           c["use_norm"], c["use_RTE"])
    m.load_state_dict(fx["state_dict"])
    return m.to(dev).eval()


def _run(m, fx, dev, key="node_inp"):
    with torch.no_grad():
        out = m(fx[key].to(dev), fx["node_type"].to(dev), fx["edge_index"].to(dev), fx["edge_type"].to(dev),
                fx["edge_time"].to(dev))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("variant", [1, 2])
@pytest.mark.parametrize("name", CONV_FIXTURES)
def test_forward_matches_reference_golden(name, variant, fused):
    """fused=True: the whole layer through ONE C-ABI call (hgt_conv_forward); False: the per-stage entry points."""
    dev = _dev()
    fx = load_golden(name)
    m = _module_from_fixture(fx, dev)
    m.edge_variant = variant
    m.fused_call = fused
    out = _run(m, fx, dev)
    _close(out, fx["out"], "%s out (variant %d, fused %s)" % (name, variant, fused))
    _close(m.att, fx["att"], "%s att (variant %d, fused %s)" % (name, variant, fused), atol=1e-4)


def test_four_argument_forward_without_rte():
    dev = _dev()
    fx = load_golden("c1_norte")
    m = _module_from_fixture(fx, dev)
    with torch.no_grad():
        out = m(fx["node_inp"].to(dev), fx["node_type"].to(dev), fx["edge_index"].to(dev), fx["edge_type"].to(dev))
    _close(out, fx["out"], "4-arg forward")


def test_plan_is_bit_exact():
    from pyhgt_b200 import plan as P
    dev = _dev()
    g = synth.make_random(5000, 40000, 5, 7, seed=3, isolated_frac=0.2, self_loops=100, duplicate_edges=500)
    nt, ei, et, tm = g.node_type, g.edge_index, g.edge_type, g.edge_time
    plan = P.build_plan(nt.to(dev), ei.to(dev), et.to(dev), tm.to(dev), g.num_types, g.num_relations)
    perm = torch.argsort(nt, stable=True)
    assert torch.equal(plan.perm.cpu().long(), perm)
    rank = torch.empty_like(perm); rank[perm] = torch.arange(perm.numel())
    assert torch.equal(plan.rank.cpu().long(), rank)
    dst_rank = rank[ei[1]]
    order = torch.argsort(dst_rank, stable=True)
    assert torch.equal(plan.csr_eid.cpu().long(), order)
    counts = torch.bincount(dst_rank, minlength=g.num_nodes)
    row_ptr = torch.cat([torch.zeros(1, dtype=torch.long), counts.cumsum(0)])
    assert torch.equal(plan.row_ptr.cpu().long(), row_ptr)
    # gather rows: pair (src_type, rel) -> base + rank-in-type
    type_count = torch.bincount(nt, minlength=g.num_types)
    type_row0 = torch.cat([torch.zeros(1, dtype=torch.long), type_count.cumsum(0)])
    pair_id = {p: i for i, p in enumerate(plan.pairs)}
    src_t = nt[ei[0]]
    exp_pairs = sorted(set(zip(src_t.tolist(), et.tolist())))
    assert plan.pairs == exp_pairs
    e_sorted = order
    exp_row = torch.tensor([plan.pair_row0[pair_id[(int(src_t[e]), int(et[e]))]] +
                            int(rank[ei[0, e]] - type_row0[src_t[e]]) for e in e_sorted.tolist()])
    assert torch.equal(plan.kv_row.cpu().long(), exp_row)
    exp_rte = torch.tensor([pair_id[(int(src_t[e]), int(et[e]))] * 240 + int(tm[e]) for e in e_sorted.tolist()])
    assert torch.equal(plan.rte_row.cpu().long(), exp_rte)
    # tiles cover every destination and every edge exactly once, in order
    tiles = plan.tiles.cpu()[:plan.n_tiles].tolist()
    d, e = 0, 0
    for t in tiles:
        if t[1] >= 0:
            assert t[0] == d and t[2] == e and t[3] == int(row_ptr[t[1]])
            d, e = t[1], t[3]
        else:
            assert t[0] == d or t[0] == d - 1
            assert t[2] == e
            e = t[3]
            d = t[0] + 1
    assert d == g.num_nodes and e == g.num_edges


def test_invalid_indices_raise():
    from pyhgt_b200 import plan as P
    dev = _dev()
    g = synth.make_c1()
    bad = g.edge_index.clone(); bad[0, 5] = g.num_nodes
    with pytest.raises(IndexError):
        P.build_plan(g.node_type.to(dev), bad.to(dev), g.edge_type.to(dev), None, 2, 1)
    tm = g.edge_time.clone(); tm[3] = 240
    with pytest.raises(IndexError):
        P.build_plan(g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev), tm.to(dev), 2, 1)
    with pytest.raises(ValueError):
        P.build_plan(g.node_type.to(dev), g.edge_index.to(dev).int(), g.edge_type.to(dev), None, 2, 1)


def test_out_of_range_relation_and_type_follow_reference_semantics():
    """Edges whose relation (or endpoint type) matches no <s,t,r> triple keep score 0 / message 0 but still
    take part in the destination's softmax (conv.py:68-69,108); nodes of unknown type get zero rows (conv.py:120)."""
    import pyhgt_b200
    dev = _dev()
    g = synth.make_random(300, 3000, 3, 4, seed=9)
    g.edge_type[::7] = 9           # relation outside [0,R)
    g.node_type[::11] = 5          # type outside [0,T)
    torch.manual_seed(1)
    m = pyhgt_b200.HGTConv(32, 32, 3, 4, 4, 0.2, True, True).eval()
    x = torch.randn(300, 32)
    params = {k: v.detach().clone() for k, v in m.state_dict().items()}
    ref, ref_att = hgt_oracle.hgt_forward_ref_port(params, x, g.node_type, g.edge_index, g.edge_type, g.edge_time,
                                                   num_types=3, num_relations=4, n_heads=4)
    m = m.to(dev)
    with torch.no_grad():
        out = m(x.to(dev), g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev), g.edge_time.to(dev))
    _close(out, ref, "out with unmatched edges")
    _close(m.att, ref_att, "att with unmatched edges", atol=1e-4)


def test_typed_linear_simt_matches_torch():
    import numpy as np
    from pyhgt_b200 import _lib, plan as P
    dev = _dev()
    torch.manual_seed(0)
    K, width = 100, 36
    a = torch.randn(777, K, device=dev)
    w = torch.randn(3 * width, K, device=dev)
    b = torch.randn(3 * width, device=dev)
    out = torch.zeros(777 * width + 500 * 2 * width, device=dev)
    # group 0: rows 0..499 -> two blocks interleaved [500, 2*width] at offset 777*width ; group 1: rows 500..776 -> block 0
    groups = [(0, 500, width, 2, 0, 1), (500, 277, 0, 1, 2, 0)]
    cblocks = [(777 * width, 2 * width), (777 * width + width, 2 * width), (500 * width, width)]
    g_dev, g_host, n_g, c_dev = P._pack_groups(groups, cblocks, dev)
    _lib.call("hgt_typed_linear", a.data_ptr(), K, w.data_ptr(), b.data_ptr(), K, width, g_dev.data_ptr(),
              g_host.ctypes.data, n_g, c_dev.data_ptr(), out.data_ptr(), 1, None, 0,
              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ref0 = a[:500].double() @ w[width:].double().t() + b[width:].double()
    got0 = out[777 * width:].view(500, 2 * width)
    assert torch.allclose(got0.double(), ref0, rtol=1e-5, atol=1e-4)
    ref1 = a[500:].double() @ w[:width].double().t()
    got1 = out[500 * width:777 * width].view(277, width)
    assert torch.allclose(got1.double(), ref1, rtol=1e-5, atol=1e-4)


def test_edge_order_permutation_invariance():
    """Permuting the edge list permutes att rows and leaves out unchanged (to fp tolerance)."""
    dev = _dev()
    fx = load_golden("rand_t3r4_dk4")
    m = _module_from_fixture(fx, dev)
    out = _run(m, fx, dev)
    att = m.att.clone()
    perm = torch.randperm(fx["edge_type"].numel(), generator=torch.Generator().manual_seed(0))
    fx2 = dict(fx)
    fx2["edge_index"] = fx["edge_index"][:, perm]
    fx2["edge_type"] = fx["edge_type"][perm]
    fx2["edge_time"] = fx["edge_time"][perm]
    out2 = _run(m, fx2, dev)
    _close(out2, out, "out under edge permutation", atol=1e-5)
    _close(m.att, att[perm.to(dev)], "att under edge permutation", atol=1e-6)


def test_empty_edge_list_gives_bias_path():
    import pyhgt_b200
    dev = _dev()
    torch.manual_seed(0)
    m = pyhgt_b200.HGTConv(32, 32, 2, 2, 4, 0.2, True, False).to(dev).eval()
    x = torch.randn(50, 32, device=dev)
    nt = torch.randint(0, 2, (50,), device=dev)
    with torch.no_grad():
        out = m(x, nt, torch.zeros(2, 0, dtype=torch.long, device=dev), torch.zeros(0, dtype=torch.long, device=dev))
    # agg = 0 -> gelu(0) = 0 -> a_linear gives its bias (SURVEY §8 a7)
    ref = torch.empty_like(out)
    for t in range(2):
        sel = nt == t
        a = torch.sigmoid(m.skip[t])
        y = m.a_linears[t].bias * a + x[sel] * (1 - a)
        ref[sel] = torch.nn.functional.layer_norm(y, (32,), m.norms[t].weight, m.norms[t].bias, 1e-5)
    _close(out, ref, "empty edge list")
    assert m.att.shape == (0, 4)


@pytest.mark.parametrize("variant", [1, 2])
def test_mag_shaped_medium_graph_vs_oracle(variant):
    """ogbn-mag-shaped graph at 0.5 % scale (~105k edges, d=256, H=8): CUDA vs CPU oracle."""
    import pyhgt_b200
    dev = _dev()
    g = synth.make_mag_shaped(scale=0.005, seed=7)
    torch.manual_seed(3)
    m = pyhgt_b200.HGTConv(256, 256, 4, 4, 8, 0.2, True, False).eval()
    x = torch.randn(g.num_nodes, 256)
    params = {k: v.detach().clone() for k, v in m.state_dict().items()}
    ref, ref_att = hgt_oracle.hgt_forward_ref_port(params, x, g.node_type, g.edge_index, g.edge_type, None,
                                                   num_types=4, num_relations=4, n_heads=8, use_RTE=False)
    m = m.to(dev)
    m.edge_variant = variant
    with torch.no_grad():
        out = m(x.to(dev), g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev))
    _close(out, ref, "mag x0.005 out")
    _close(m.att, ref_att, "mag x0.005 att", atol=1e-4)


def test_hub_split_matches_unsplit(monkeypatch):
    """Force hub splitting at a tiny threshold: result must not change."""
    from pyhgt_b200 import plan as P
    dev = _dev()
    fx = load_golden("hub_h2")
    m = _module_from_fixture(fx, dev)
    out_ref = _run(m, fx, dev)
    att_ref = m.att.clone()
    monkeypatch.setattr(P, "TILE_SPLIT_EDGES", 37)
    monkeypatch.setattr(P, "TILE_TARGET_EDGES", 8)
    P.clear_plan_cache()
    for variant in (1, 2):
        m.edge_variant = variant
        fx2 = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in fx.items()}
        out = _run(m, fx2, dev)
        _close(out, out_ref, "hub split out (variant %d)" % variant, atol=1e-5)
        _close(m.att, att_ref, "hub split att", atol=1e-6)
        _close(out, fx["out"], "hub split vs golden")
    P.clear_plan_cache()


@pytest.mark.parametrize("K,width,m_rows", [(256, 256, 1000), (64, 64, 130), (400, 400, 300), (128, 48, 257), (104, 32, 64)])
def test_typed_linear_tensor_core_matches_fp64(K, width, m_rows):
    """tcgen05 split-bf16 GEMM (impl 2) against float64: error must be ~1e-5 relative, far inside 1e-3."""
    import ctypes
    from pyhgt_b200 import _lib, plan as P
    dev = _dev()
    torch.manual_seed(K + width)
    a = torch.randn(m_rows + 77, K, device=dev)
    w = torch.randn(3 * width, K, device=dev) / K ** 0.5
    b = torch.randn(3 * width, device=dev)
    out = torch.full((m_rows * width + 77 * 2 * width,), float("nan"), device=dev)
    groups = [(0, m_rows, 0, 1, 0, 1), (m_rows, 77, width, 2, 1, 0)]
    cblocks = [(0, width), (m_rows * width, 2 * width), (m_rows * width + width, 2 * width)]
    g_dev, g_host, n_g, c_dev = P._pack_groups(groups, cblocks, dev)
    ws_bytes = ctypes.c_size_t()
    _lib.call("hgt_typed_linear_workspace_bytes", g_host.ctypes.data, n_g, K, width, 2, ctypes.byref(ws_bytes))
    ws = torch.empty(max(ws_bytes.value, 1), dtype=torch.uint8, device=dev)
    _lib.call("hgt_typed_linear", a.data_ptr(), K, w.data_ptr(), b.data_ptr(), K, width, g_dev.data_ptr(),
              g_host.ctypes.data, n_g, c_dev.data_ptr(), out.data_ptr(), 2, ws.data_ptr(), ws.numel(),
              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ref0 = a[:m_rows].double() @ w[:width].double().t() + b[:width].double()
    got0 = out[:m_rows * width].view(m_rows, width).double()
    ref1 = a[m_rows:].double() @ w[width:].double().t()
    got1 = out[m_rows * width:].view(77, 2 * width).double()
    for got, ref in ((got0, ref0), (got1, ref1)):
        assert torch.isfinite(got).all()
        err = (got - ref).abs().max().item()
        assert err < 5e-5 * max(1.0, ref.abs().max().item()), "max abs err %.3g" % err


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_local_forward_matches_full_graph(world):
    """The kernels on one rank's shard (owned + halo rows, Q/update restricted to owned rows) reproduce the
    full-graph result on the owned rows.  The halo exchange itself is covered by tests/test_sharded_cpu.py."""
    import pyhgt_b200
    from pyhgt_b200 import sharded
    dev = _dev()
    g = synth.make_random(900, 9000, 3, 4, seed=11, isolated_frac=0.2, self_loops=60, duplicate_edges=90)
    torch.manual_seed(5)
    m = pyhgt_b200.HGTConv(64, 64, 3, 4, 4, 0.2, True, True).to(dev).eval()
    x = torch.randn(g.num_nodes, 64)
    with torch.no_grad():
        full = m(x.to(dev), g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev), g.edge_time.to(dev)).cpu()
    for rank in range(world):
        sh = sharded.ShardedGraph.build(g.node_type, g.edge_index, g.edge_type, g.edge_time, 3, 4, rank, world, dev)
        x_local = x[sh.local_global].to(dev)
        assert torch.all(sh.node_type[1:] >= sh.node_type[:-1])          # local order is type-sorted
        with torch.no_grad():
            out, _, _ = m._forward_impl(x_local, sh.node_type, sh.edge_index, sh.edge_type, sh.edge_time,
                                        want_att=False, save=False, active_per_type=sh.active_per_type)
        _close(out[sh.own_rows], full[sh.owned_global], "rank %d/%d owned rows" % (rank, world), atol=1e-5)
        # ShardedGraph.forward's direct-to-owned-order epilogue (world=1 exchange is the identity gather)
        om = torch.full((sh.n_owned + sh.n_halo,), -1, dtype=torch.int32, device=dev)
        om[sh.own_rows] = torch.arange(sh.n_owned, dtype=torch.int32, device=dev)
        with torch.no_grad():
            out2, _, _ = m._forward_impl(x_local, sh.node_type, sh.edge_index, sh.edge_type, sh.edge_time,
                                         want_att=False, save=False, active_per_type=sh.active_per_type,
                                         out_map=om, out_rows=sh.n_owned)
        _close(out2, full[sh.owned_global], "rank %d/%d direct owned-order output" % (rank, world), atol=1e-5)
        # per-pair compaction (what ShardedGraph.forward ships): K'/V' projected only for the row ranges local edges read
        assert sh.kv_runs is not None
        from pyhgt_b200 import plan as P
        pl = P.get_plan(sh.node_type, sh.edge_index, sh.edge_type, sh.edge_time, 3, 4)
        full_rows = sum(pl.type_count[s_] for (s_, _) in pl.pairs)
        run_rows = sum(r1 - r0 for (key, rs) in sh.kv_runs if key in pl.pairs for (r0, r1) in rs)
        assert run_rows < full_rows
        for fused in (True, False):
            m.fused_call = fused
            with torch.no_grad():
                out3, _, _ = m._forward_impl(x_local, sh.node_type, sh.edge_index, sh.edge_type, sh.edge_time,
                                             want_att=False, save=False, active_per_type=sh.active_per_type,
                                             out_map=om, out_rows=sh.n_owned, kv_runs=sh.kv_runs)
            _close(out3, full[sh.owned_global], "rank %d/%d compacted projection (fused %s)" % (rank, world, fused),
                   atol=1e-5)
        m.fused_call = True


@pytest.mark.parametrize("name", ["c1_rte", "rand_t3r4_dk4"])
def test_backward_matches_reference_autograd(name):
    """d(sum(out*w))/d{node_inp, every parameter} against the gradients the reference's own autograd produced
    (tests/golden, oracle/make_golden.py)."""
    dev = _dev()
    fx = load_golden(name)
    m = _module_from_fixture(fx, dev)      # eval(): dropout off, same as the fixture
    x = fx["node_inp"].to(dev).requires_grad_(True)
    out = m(x, fx["node_type"].to(dev), fx["edge_index"].to(dev), fx["edge_type"].to(dev), fx["edge_time"].to(dev))
    _close(out.detach(), fx["out"], name + " training-path out")
    _close(m.att, fx["att"], name + " training-path att", atol=1e-4)
    (out * fx["grad_weight"].to(dev)).sum().backward()

    def check(got, ref, what):
        got, ref = got.float().cpu(), ref.float()
        scale = ref.abs().max().item()
        fro = ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()
        assert torch.allclose(got, ref, rtol=1e-3, atol=1e-3 * max(scale, 1e-6)), \
            "%s: max abs err %.3g (scale %.3g, rel fro %.3g)" % (what, (got - ref).abs().max().item(), scale, fro)
        assert fro <= 2e-3, "%s: relative Frobenius error %.3g" % (what, fro)

    check(x.grad, fx["grad_node_inp"], name + " d node_inp")
    got = {k: p.grad for k, p in m.named_parameters()}
    for k, ref in fx["grad_params"].items():
        assert got[k] is not None, "no gradient for %s" % k
        check(got[k], ref, name + " d " + k)


def test_backward_hub_split_and_unsorted_types():
    """Gradients with hub splitting forced (atomic dq path) equal the unsplit ones; compared against autograd
    through the CPU oracle port."""
    import pyhgt_b200
    from pyhgt_b200 import plan as P
    dev = _dev()
    g = synth.make_random(200, 1500, 2, 3, seed=31)
    hub = torch.full((600,), 5, dtype=torch.int64)
    gen = torch.Generator().manual_seed(3)
    g.edge_index = torch.cat([g.edge_index, torch.stack([torch.randint(0, 200, (600,), generator=gen), hub])], 1)
    g.edge_type = torch.cat([g.edge_type, torch.randint(0, 3, (600,), generator=gen)])
    g.edge_time = torch.cat([g.edge_time, torch.randint(0, 240, (600,), generator=gen)])
    torch.manual_seed(2)
    m = pyhgt_b200.HGTConv(32, 32, 2, 3, 4, 0.0, True, True).eval()
    x = torch.randn(200, 32)
    w = torch.randn(200, 32)
    params = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    xr = x.clone().requires_grad_(True)
    ref, _ = hgt_oracle.hgt_forward_ref_port(params, xr, g.node_type, g.edge_index, g.edge_type, g.edge_time,
                                             num_types=2, num_relations=3, n_heads=4)
    (ref * w).sum().backward()
    m = m.to(dev)
    old = (P.TILE_SPLIT_EDGES, P.TILE_TARGET_EDGES)
    try:
        P.TILE_SPLIT_EDGES, P.TILE_TARGET_EDGES = 50, 8
        P.clear_plan_cache()
        xg = x.to(dev).requires_grad_(True)
        out = m(xg, g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev), g.edge_time.to(dev))
        (out * w.to(dev)).sum().backward()
    finally:
        P.TILE_SPLIT_EDGES, P.TILE_TARGET_EDGES = old
        P.clear_plan_cache()
    _close(out.detach(), ref.detach(), "hub training out")
    for got, exp, what in [(xg.grad, xr.grad, "d node_inp")] + \
            [(p.grad, params[k].grad, "d " + k) for k, p in m.named_parameters() if params[k].grad is not None]:
        got, exp = got.cpu(), exp
        scale = max(exp.abs().max().item(), 1e-6)
        assert torch.allclose(got, exp, rtol=2e-3, atol=2e-3 * scale), \
            "%s: max abs err %.3g (scale %.3g)" % (what, (got - exp).abs().max().item(), scale)


def test_gnn_stack_matches_reference_model_golden():
    """pyhgt_b200.model.GNN (adapter + 2 HGT layers, one shared plan) against the reference's model.py output."""
    from pyhgt_b200.model import GNN
    dev = _dev()
    fx = load_golden("gnn_2layer")
    c = fx["cfg"]
    m = GNN(c["in_dim"], c["n_hid"], c["num_types"], c["num_relations"], c["n_heads"], c["n_layers"], 0.2, "hgt",
            c["prev_norm"], c["last_norm"], c["use_RTE"])
    m.load_state_dict(fx["state_dict"], strict=True)
    m = m.to(dev).eval()
    with torch.no_grad():
        out = m(fx["node_feature"].to(dev), fx["node_type"].to(dev), fx["edge_time"].to(dev),
                fx["edge_index"].to(dev), fx["edge_type"].to(dev))
    _close(out, fx["out"], "GNN 2-layer out")


def test_dense_hgt_conv_matches_reference_golden():
    """DenseHGTConv (conv.py:143-280) — same message kernels, residual/LayerNorm/FFN update."""
    import pyhgt_b200
    dev = _dev()
    fx = load_golden("dense_hgt")
    c = fx["cfg"]
    g = pyhgt_b200.GeneralConv('dense_hgt', c["in_dim"], c["out_dim"], c["num_types"], c["num_relations"], c["n_heads"],
                               0.2, c["use_norm"], c["use_RTE"])
    m = g.base_conv
    m.load_state_dict(fx["state_dict"], strict=True)
    g = g.to(dev).eval()
    with torch.no_grad():
        out = g(fx["node_inp"].to(dev), fx["node_type"].to(dev), fx["edge_index"].to(dev), fx["edge_type"].to(dev),
                fx["edge_time"].to(dev))
    _close(out, fx["out"], "dense_hgt out")
    _close(m.att, fx["att"], "dense_hgt att", atol=1e-4)


def test_full_size_c2_properties_and_sampled_rows():
    """BASELINE config 2 at FULL size (1.94 M nodes, 21.1 M edges, d=256): (a) the output rows of 3000 sampled
    destinations equal the CPU oracle run on their 1-hop induced subgraph (a destination's row depends only on its
    in-edges and their sources), (b) per-destination attention sums to 1, (c) isolated destinations take the
    bias path, (d) both edge-kernel variants agree."""
    import pyhgt_b200
    dev = _dev()
    g = synth.make_mag_shaped(1.0, seed=2)
    N, E, d, H = g.num_nodes, g.num_edges, 256, 8
    torch.manual_seed(0)
    m = pyhgt_b200.HGTConv(d, d, 4, 4, H, 0.2, True, False).eval()
    x = torch.randn(N, d, generator=torch.Generator().manual_seed(1))
    params = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.to(dev)
    nt, ei, et = g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev)
    xd = x.to(dev)
    old_keep = pyhgt_b200.HGTConv.keep_att
    try:
        pyhgt_b200.HGTConv.keep_att = True
        with torch.no_grad():
            m.edge_variant = 2
            out = m(xd, nt, ei, et)
            att = m.att
            sums = torch.zeros(N, H, device=dev).index_add_(0, ei[1], att)
            deg = torch.bincount(ei[1], minlength=N)
            assert torch.allclose(sums[deg > 0], torch.ones_like(sums[deg > 0]), atol=1e-4)
            assert torch.all(sums[deg == 0] == 0)
            del att, sums
            pyhgt_b200.HGTConv.keep_att = False
            m.edge_variant = 1
            out1 = m(xd, nt, ei, et)
        assert torch.isfinite(out).all()
        _close(out1, out, "variant 1 vs 2 at full size", atol=1e-5)
        del out1
    finally:
        pyhgt_b200.HGTConv.keep_att = old_keep
    # (a) sampled destinations vs the oracle on the induced 1-hop subgraph
    gen = torch.Generator().manual_seed(5)
    has_in = (deg > 0).cpu().nonzero(as_tuple=True)[0]
    sample = torch.cat([has_in[torch.randperm(has_in.numel(), generator=gen)[:2500]],
                        (deg == 0).cpu().nonzero(as_tuple=True)[0][:500]])
    sel = torch.zeros(N, dtype=torch.bool); sel[sample] = True
    e_sel = sel[g.edge_index[1]].nonzero(as_tuple=True)[0]
    nodes = torch.unique(torch.cat([sample, g.edge_index[0, e_sel]]))
    local = torch.full((N,), -1, dtype=torch.int64); local[nodes] = torch.arange(nodes.numel())
    sub_ei = torch.stack([local[g.edge_index[0, e_sel]], local[g.edge_index[1, e_sel]]])
    ref, _ = hgt_oracle.hgt_forward_ref_port(params, x[nodes], g.node_type[nodes], sub_ei, g.edge_type[e_sel], None,
                                             num_types=4, num_relations=4, n_heads=H, use_norm=True, use_RTE=False)
    _close(out[sample.to(dev)], ref[local[sample]], "full-size C2: sampled destination rows vs oracle")


def test_to_torch_device_ingest_prebuilds_plan():
    """pyhgt_b200.data.to_torch(device=cuda, prebuild_plan=True): tensors arrive on the GPU and the layer reuses the plan."""
    import pyhgt_b200
    from pyhgt_b200 import data as hdata, plan as P
    from tests.test_data_ingest import _GraphStub
    dev = _dev()
    fx = load_golden("to_torch")
    g = _GraphStub(fx["types"], fx["meta_graph"])
    P.clear_plan_cache()
    nf, nt, etime, ei, et, node_dict, edge_dict = hdata.to_torch(fx["feature"], fx["time"], fx["edge_list"], g,
                                                                device=dev, prebuild_plan=True)
    assert nf.is_cuda and ei.is_cuda and torch.equal(ei.cpu(), fx["edge_index"])
    assert len(P._CACHE) == 1
    d = nf.shape[1]
    torch.manual_seed(0)
    # d = 7 is odd: the reference's RelTemporalEncoding cannot even be built for odd widths (conv.py:293-294), so the
    # layer runs without RTE; it also exercises the scalar (VEC = 1) lane mapping and the fp32 SIMT GEMM.
    m = pyhgt_b200.HGTConv(d, d, len(fx["types"]), len(edge_dict), 1, 0.2, True, False).to(dev).eval()
    P.clear_plan_cache()
    P.get_plan(nt, ei, et, None, len(fx["types"]), len(edge_dict))
    with torch.no_grad():
        out = m(nf, nt, ei, et, etime)
    assert len(P._CACHE) == 1 and torch.isfinite(out).all()       # same tensors -> cached plan reused
    params = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    ref, _ = hgt_oracle.hgt_forward_ref_port(params, fx["node_feature"], fx["node_type"], fx["edge_index"],
                                             fx["edge_type"], None, num_types=len(fx["types"]),
                                             num_relations=len(edge_dict), n_heads=1, use_RTE=False)
    _close(out, ref, "layer on to_torch output")


def _sampled_rows_vs_oracle(g, d, H, rte, n_with=1200, n_isolated=200, seed=5, variant=0, what=""):
    """Full-size technique (SURVEY.md §8d): the output rows of sampled destinations equal the CPU oracle run on their
    1-hop induced subgraph, because a destination's row depends only on its in-edges and their sources."""
    import pyhgt_b200
    dev = _dev()
    N = g.num_nodes
    T, R = g.num_types, g.num_relations
    torch.manual_seed(0)
    m = pyhgt_b200.HGTConv(d, d, T, R, H, 0.2, True, rte).eval()
    x = torch.randn(N, d, generator=torch.Generator().manual_seed(1))
    params = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.to(dev)
    m.edge_variant = variant
    old_keep = pyhgt_b200.HGTConv.keep_att
    try:
        pyhgt_b200.HGTConv.keep_att = False
        with torch.no_grad():
            out = m(x.to(dev), g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev),
                    g.edge_time.to(dev) if rte else None)
    finally:
        pyhgt_b200.HGTConv.keep_att = old_keep
    assert torch.isfinite(out).all()
    deg = torch.bincount(g.edge_index[1], minlength=N)
    gen = torch.Generator().manual_seed(seed)
    has_in = (deg > 0).nonzero(as_tuple=True)[0]
    # always include the heaviest destinations (hub splitting / merge path)
    hubs = torch.argsort(deg, descending=True)[:8]
    sample = torch.unique(torch.cat([has_in[torch.randperm(has_in.numel(), generator=gen)[:n_with]], hubs,
                                     (deg == 0).nonzero(as_tuple=True)[0][:n_isolated]]))
    sel = torch.zeros(N, dtype=torch.bool); sel[sample] = True
    e_sel = sel[g.edge_index[1]].nonzero(as_tuple=True)[0]
    nodes = torch.unique(torch.cat([sample, g.edge_index[0, e_sel]]))
    local = torch.full((N,), -1, dtype=torch.int64); local[nodes] = torch.arange(nodes.numel())
    sub_ei = torch.stack([local[g.edge_index[0, e_sel]], local[g.edge_index[1, e_sel]]])
    ref, _ = hgt_oracle.hgt_forward_ref_port(params, x[nodes], g.node_type[nodes], sub_ei, g.edge_type[e_sel],
                                             g.edge_time[e_sel] if rte else None, num_types=T, num_relations=R,
                                             n_heads=H, use_norm=True, use_RTE=rte)
    _close(out[sample.to(dev)], ref[local[sample]], what + ": sampled destination rows vs oracle")
    return int(deg.max())


def test_full_size_c3_sampled_rows():
    """BASELINE config 3 at FULL size: OAG-CS-shaped, 6 types / 10 relations incl. `self`, N=200 k, E=5 M, d=400
    (d_k=50: the VEC=2 lane map), RTE on."""
    g = synth.make_oag_shaped(1.0)
    assert g.num_edges >= 4_900_000 and g.num_types == 6 and g.num_relations == 10
    _sampled_rows_vs_oracle(g, 400, 8, True, n_with=600, n_isolated=0, what="full-size C3")


def test_full_size_c5_16m_sampled_rows_including_hubs():
    """BASELINE config 5 (16 M-edge member): power-law destinations, thousands of hub pieces merged by k_merge_partials;
    the sample always contains the 8 heaviest destinations."""
    g = synth.make_powerlaw(16_000_000)
    max_deg = _sampled_rows_vs_oracle(g, 128, 8, False, n_with=800, n_isolated=100, what="C5-16M")
    assert max_deg > 1024                                   # the hub path was exercised


def test_typed_linear_more_groups_than_one_launch_holds():
    """Schemas with > 64 <type, relation> groups (ADVICE r1): the entry point launches in chunks.  The second shape,
    K = 2304, leaves no room for a resident W tile, so the tensor-core path takes the one-tile-per-CTA kernel."""
    import ctypes
    import re
    from torch.profiler import profile, ProfilerActivity
    from pyhgt_b200 import _lib, plan as P
    dev = _dev()
    for K, width, n_g, m in ((64, 32, 70, 37), (2304, 256, 2, 300)):
        gen = torch.Generator().manual_seed(0)
        A = torch.randn(n_g * m, K, generator=gen)
        W = torch.randn(n_g * width, K, generator=gen)
        b = torch.randn(n_g * width, generator=gen)
        groups = [(i * m, m, i * width, 1, i, 1) for i in range(n_g)]
        cblocks = [(i * m * width, width) for i in range(n_g)]
        for impl in (1, 2):
            tab = P._pack_groups(groups, cblocks, dev)
            out = torch.zeros(n_g * m * width, device=dev)
            wsb = ctypes.c_size_t()
            _lib.call("hgt_typed_linear_workspace_bytes", tab[1].ctypes.data, n_g, K, width, impl, ctypes.byref(wsb))
            ws = torch.empty(max(wsb.value, 1), dtype=torch.uint8, device=dev)
            Ad, Wd, bd = A.to(dev), W.to(dev), b.to(dev)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                _lib.call("hgt_typed_linear", Ad.data_ptr(), K, Wd.data_ptr(), bd.data_ptr(), K, width,
                          tab[0].data_ptr(), tab[1].ctypes.data, n_g, tab[3].data_ptr(), out.data_ptr(), impl,
                          ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
            ref = torch.stack([A[i * m:(i + 1) * m].double() @ W[i * width:(i + 1) * width].double().t()
                               + b[i * width:(i + 1) * width].double() for i in range(n_g)]).float()
            _close(out.view(n_g, m, width), ref, "typed linear, K=%d, %d groups, impl %d" % (K, n_g, impl))
            if impl == 2 and K > 2240:
                names = [e.key for e in prof.key_averages()]
                assert any(re.search(r"k_typed_linear_tc(?![23])", n) for n in names), names


def test_backward_two_graphs_same_pairs_no_stale_tables():
    """ADVICE r1 (high): a sampled-subgraph loop builds a new plan per batch; the backward of the second graph must use
    ITS column-block table even when the pair set is identical and the plan cache was cleared in between."""
    import pyhgt_b200
    from pyhgt_b200 import plan as P
    dev = _dev()
    torch.manual_seed(0)
    m = pyhgt_b200.HGTConv(64, 64, 3, 2, 4, 0.0, True, False).to(dev).train()
    params = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    old_keep = pyhgt_b200.HGTConv.keep_att
    pyhgt_b200.HGTConv.keep_att = False
    try:
        for seed, n in ((1, 300), (2, 517)):                     # same <type, relation> pairs, different type counts
            g = synth.make_random(n, 4 * n, 3, 2, seed=seed, sorted_types=True)
            x = torch.randn(n, 64, generator=torch.Generator().manual_seed(seed))
            xd = x.to(dev).requires_grad_(True)
            P.clear_plan_cache()
            out = m(xd, g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev))
            w = torch.randn(n, 64, generator=torch.Generator().manual_seed(9))
            (out * w.to(dev)).sum().backward()
            xr = x.clone().requires_grad_(True)
            for v in params.values():
                v.grad = None
            ref, _ = hgt_oracle.hgt_forward_ref_port(params, xr, g.node_type, g.edge_index, g.edge_type, None,
                                                     num_types=3, num_relations=2, n_heads=4, use_norm=True,
                                                     use_RTE=False)
            (ref * w).sum().backward()
            _close(out.detach(), ref.detach(), "graph %d out" % seed)
            for got, exp, what in [(xd.grad, xr.grad, "d node_inp")] + \
                    [(p.grad, params[k].grad, "d " + k) for k, p in m.named_parameters() if params[k].grad is not None]:
                got = got.cpu()
                scale = max(exp.abs().max().item(), 1e-6)
                assert torch.allclose(got, exp, rtol=2e-3, atol=2e-3 * scale), \
                    "graph %d %s: max abs err %.3g (scale %.3g)" % (seed, what, (got - exp).abs().max().item(), scale)
            m.zero_grad()
    finally:
        pyhgt_b200.HGTConv.keep_att = old_keep


def test_module_saves_after_inference_forward(tmp_path):
    """torch.save(model) after an eval pass, then load and run again (OAG/train_paper_field.py:279,311)."""
    import pyhgt_b200
    dev = _dev()
    fx = load_golden("c1_rte")
    m = _module_from_fixture(fx, dev)
    out = _run(m, fx, dev)
    path = tmp_path / "model.pt"
    torch.save(m, path)
    m2 = torch.load(path, weights_only=False).to(dev).eval()
    out2 = _run(m2, fx, dev)
    assert torch.equal(out, out2)
    _close(out2, fx["out"], "reloaded module")


def test_sampled_subgraph_batch_runs_without_host_sync():
    """The reference's training regime (OAG/train_paper_field.py:241): a NEW sampled graph every batch.  After a warm-up,
    `to_torch(device=cuda, prebuild_plan=True)` + the layer run with NO host synchronisation (torch's sync debug mode
    raises on any blocking call) and the sync-free plan gives the same result as the synchronous one and the oracle."""
    import pyhgt_b200
    from pyhgt_b200 import data as hdata, plan as P
    from tests.test_data_ingest import _GraphStub
    dev = _dev()
    fx = load_golden("to_torch")
    g = _GraphStub(fx["types"], fx["meta_graph"])
    T = len(fx["types"])
    d = fx["node_feature"].shape[1]
    torch.manual_seed(0)
    m = None

    def batch():
        nf, nt, etime, ei, et, node_dict, edge_dict = hdata.to_torch(fx["feature"], fx["time"], fx["edge_list"], g,
                                                                    device=dev, prebuild_plan=True)
        return nf, nt, etime, ei, et, len(edge_dict)

    nf, nt, etime, ei, et, R = batch()
    m = pyhgt_b200.HGTConv(d, d, T, R, 1, 0.2, True, False).to(dev).eval()
    with torch.no_grad():
        ref_sync = m(nf, nt, fx["edge_index"].to(dev), et)                 # synchronous plan (different tensor object)
        out0 = m(nf, nt, ei, et, etime)                                   # warm-up of the sync-free path
    torch.cuda.synchronize()
    pl = P.get_plan(nt, ei, et, None, T, R)              # the layer asks without edge_time (no RTE): served by the prebuilt plan
    assert pl.tile_counts_dev is not None                                 # the prebuilt plan is the sync-free one
    pl.check()
    P.clear_plan_cache()
    torch.cuda.set_sync_debug_mode("error")
    try:
        with torch.no_grad():
            nf2, nt2, etime2, ei2, et2, _ = batch()                       # new tensors => new plan
            out = m(nf2, nt2, ei2, et2, etime2)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.equal(out, out0)
    _close(out, ref_sync, "sync-free plan vs synchronous plan", atol=1e-6)
    params = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    ref, _ = hgt_oracle.hgt_forward_ref_port(params, fx["node_feature"], fx["node_type"], fx["edge_index"],
                                             fx["edge_type"], None, num_types=T, num_relations=R, n_heads=1,
                                             use_RTE=False)
    _close(out, ref, "sync-free batch vs oracle")


def test_sync_free_plan_with_hubs_matches_synchronous_plan():
    """Device-side tile counts (upper-bound grids, hub merge bounded on the device) on a graph with split hubs, forward
    and backward."""
    import pyhgt_b200
    from pyhgt_b200 import plan as P
    dev = _dev()
    g = synth.make_random(600, 3000, 3, 2, seed=41, sorted_types=True)
    gen = torch.Generator().manual_seed(4)
    hub = torch.full((2500,), 17, dtype=torch.int64)
    g.edge_index = torch.cat([g.edge_index, torch.stack([torch.randint(0, 600, (2500,), generator=gen), hub])], 1)
    g.edge_type = torch.cat([g.edge_type, torch.randint(0, 2, (2500,), generator=gen)])
    torch.manual_seed(1)
    m = pyhgt_b200.HGTConv(64, 64, 3, 2, 4, 0.0, True, False).to(dev).eval()
    x = torch.randn(600, 64, generator=torch.Generator().manual_seed(2)).to(dev)
    nt, ei, et = g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev)
    counts = torch.bincount(g.node_type, minlength=3).tolist()
    pairs = sorted({(int(g.node_type[s]), int(r)) for s, r in zip(g.edge_index[0].tolist(), g.edge_type.tolist())})
    outs, grads = [], []
    for meta in (None, {"type_count": counts + [0], "sorted": True, "pairs": pairs}):
        P.clear_plan_cache()
        pl = P.get_plan(nt, ei, et, None, 3, 2, host_meta=meta)
        assert (pl.tile_counts_dev is not None) == (meta is not None)
        if meta is not None:
            assert pl.n_hubs >= 1 and pl.n_split >= 3
        with torch.no_grad():
            outs.append(m(x, nt, ei, et).clone())
        xg = x.clone().requires_grad_(True)
        m(xg, nt, ei, et).square().sum().backward()
        grads.append(xg.grad.clone())
        m.zero_grad()
    P.clear_plan_cache()
    _close(outs[1], outs[0], "sync-free vs synchronous plan (hubs)", atol=1e-6)
    _close(grads[1], grads[0], "sync-free vs synchronous plan (hubs), d x", atol=1e-5)


def test_cuda_graph_replay_of_plan_and_layers_matches_eager():
    """graphed.GraphedForward: plan build + a 2-layer GNN captured once for a padded signature, replayed for batches of
    different sizes; every batch equals the eager result on the unpadded batch."""
    from pyhgt_b200.model import GNN
    from pyhgt_b200 import graphed
    dev = _dev()
    T, R, F_in, n_hid = 3, 4, 48, 64
    torch.manual_seed(3)
    m = GNN(F_in, n_hid, T, R, 4, 2, 0.2, "hgt", True, False, True).to(dev).eval()
    batches = [synth.make_random(n, e, T, R, seed=s, sorted_types=True, self_loops=20)
               for n, e, s in ((400, 3000, 1), (310, 2200, 2), (455, 3400, 3))]
    counts = [max(int((b.node_type == t).sum()) for b in batches) + 5 for t in range(T)]
    pairs = {(int(b.node_type[s_]), int(r_)) for b in batches for s_, r_ in zip(b.edge_index[0].tolist(), b.edge_type.tolist())}
    sig = graphed.GraphSignature(counts, 3600, pairs, R, F_in, use_time=True)
    g = graphed.GraphedForward(lambda x, nt, tm, ei, et: m(x, nt, tm, ei, et), sig, dev)
    old_keep = __import__("pyhgt_b200").HGTConv.keep_att
    __import__("pyhgt_b200").HGTConv.keep_att = False
    try:
        for rep in range(2):
            for b in batches:
                x = torch.randn(b.num_nodes, F_in, generator=torch.Generator().manual_seed(7 + b.num_nodes))
                out = g(x, b.node_type, b.edge_time, b.edge_index, b.edge_type)
                with torch.no_grad():
                    ref = m(x.to(dev), b.node_type.to(dev), b.edge_time.to(dev), b.edge_index.to(dev), b.edge_type.to(dev))
                torch.cuda.synchronize()
                _close(out, ref, "graph replay vs eager (N=%d, pass %d)" % (b.num_nodes, rep), atol=1e-5)
    finally:
        __import__("pyhgt_b200").HGTConv.keep_att = old_keep
    # a batch that does not fit is refused, not silently truncated
    big = synth.make_random(2000, 3000, T, R, seed=9, sorted_types=True)
    with pytest.raises(ValueError):
        g(torch.randn(2000, F_in), big.node_type, big.edge_time, big.edge_index, big.edge_type)
