"""Deterministic training mode (``torch.use_deterministic_algorithms(True)``): every backward stage takes its ``*_det``
entry point, so gradients repeat bit for bit from run to run; they still match the reference's autograd and, up to
summation order, the default (atomic) backward."""
import contextlib
import ctypes
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

import pyhgt_b200                                              # noqa: E402
from pyhgt_b200 import _lib, synth, plan as P                  # noqa: E402
from pyhgt_b200.model import GNN                               # noqa: E402
from oracle import hgt_oracle                                  # noqa: E402
from tests.conftest import load_golden                         # noqa: E402


def _dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _stream():
    return torch.cuda.current_stream().cuda_stream


@contextlib.contextmanager
def deterministic(on=True):
    old = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(old)


@contextlib.contextmanager
def tile_thresholds(split, target):
    old = (P.TILE_SPLIT_EDGES, P.TILE_TARGET_EDGES)
    P.TILE_SPLIT_EDGES, P.TILE_TARGET_EDGES = split, target
    P.clear_plan_cache()
    try:
        yield
    finally:
        P.TILE_SPLIT_EDGES, P.TILE_TARGET_EDGES = old
        P.clear_plan_cache()


def _rel_fro(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _check_ref(got, ref, what):
    """The bar of the existing reference-gradient tests (test_gpu_bwd.py / test_gpu_parity.py)."""
    got, ref = got.float().cpu(), ref.float()
    scale = ref.abs().max().item()
    fro = _rel_fro(got, ref)
    assert torch.allclose(got, ref, rtol=1e-3, atol=1e-3 * max(scale, 1e-6)), \
        "%s: max abs err %.3g (scale %.3g, rel fro %.3g)" % (what, (got - ref).abs().max().item(), scale, fro)
    assert fro <= 2e-3, "%s: relative Frobenius error %.3g" % (what, fro)


# ---- models built from the golden fixtures -------------------------------------------------------------------------------

def _case(name, dev):
    """(module, inputs, input-feature tensor, output weight) of a fixture; modules in eval() (dropout off)."""
    fx = load_golden(name)
    c = fx["cfg"]
    if name == "gnn_2layer":
        m = GNN(c["in_dim"], c["n_hid"], c["num_types"], c["num_relations"], c["n_heads"], c["n_layers"], 0.2, "hgt",
                c["prev_norm"], c["last_norm"], c["use_RTE"])
        x = fx["node_feature"]
        args = (fx["node_type"], fx["edge_time"], fx["edge_index"], fx["edge_type"])
    else:
        cls = pyhgt_b200.DenseHGTConv if name == "dense_hgt" else pyhgt_b200.HGTConv
        m = cls(c["in_dim"], c["out_dim"], c["num_types"], c["num_relations"], c["n_heads"], 0.2, c["use_norm"],
                c["use_RTE"])
        x = fx["node_inp"]
        args = (fx["node_type"], fx["edge_index"], fx["edge_type"], fx["edge_time"])
    m.load_state_dict(fx["state_dict"], strict=True)
    m = m.to(dev).eval()
    w = fx.get("grad_weight")
    if w is None:
        w = torch.randn(x.shape[0], m(x.to(dev), *[a.to(dev) for a in args]).shape[1],
                        generator=torch.Generator().manual_seed(7))
    return m, x.to(dev), tuple(a.to(dev) for a in args), w.to(dev), fx


def _grads(m, x, args, w):
    m.zero_grad(set_to_none=True)
    xg = x.clone().requires_grad_(True)
    out = m(xg, *args)
    (out * w).sum().backward()
    g = {"<input>": xg.grad.detach().clone()}
    for k, p in m.named_parameters():
        if p.grad is not None:
            g[k] = p.grad.detach().clone()
    return g


def _assert_bitwise(runs, what):
    ref = runs[0]
    for i, g in enumerate(runs[1:], 1):
        assert g.keys() == ref.keys()
        for k in ref:
            assert torch.isfinite(g[k]).all(), "%s: %s has non-finite entries (run %d)" % (what, k, i)
            a, b = g[k].contiguous().view(torch.int32), ref[k].contiguous().view(torch.int32)
            assert torch.equal(a, b), "%s: %s differs bitwise between runs 0 and %d (%d elements)" % (
                what, k, i, int((a != b).sum()))


def _busy_side_stream(dev):
    """Work on another stream that keeps SMs occupied while the measured step runs (changes the CTA schedule)."""
    s = torch.cuda.Stream(device=dev)
    a = torch.randn(2048, 2048, device=dev)
    with torch.cuda.stream(s):
        for _ in range(30):
            a = torch.tanh(a @ a * 1e-3)
    return s


@pytest.mark.parametrize("name", ["c1_norte", "c1_rte", "rand_t3r4_dk4", "rand_dk25", "mag_mini_dk50", "hub_h2",
                                  "dense_hgt", "gnn_2layer"])
def test_gradients_repeat_bitwise(name):
    dev = _dev()
    m, x, args, w, _ = _case(name, dev)
    runs = []
    with deterministic():
        for i in range(3):
            P.clear_plan_cache()
            side = _busy_side_stream(dev) if i == 1 else None
            runs.append(_grads(m, x, args, w))
            if side is not None:
                side.synchronize()
    P.clear_plan_cache()
    _assert_bitwise(runs, name)


def test_hub_sources_and_destinations_repeat_bitwise_and_match_oracle():
    """One source feeds 600 edges of one relation at one time offset (a hub [K'|V'] row and a hub RTE row) and one
    destination receives 600 edges, with the split threshold lowered to 50: all three indices of the deterministic
    edge backward split and merge pieces."""
    dev = _dev()
    g = synth.make_random(200, 1500, 2, 3, seed=31)
    gen = torch.Generator().manual_seed(3)
    n_hub = 600
    src_hub = torch.stack([torch.full((n_hub,), 7, dtype=torch.int64), torch.randint(0, 200, (n_hub,), generator=gen)])
    dst_hub = torch.stack([torch.randint(0, 200, (n_hub,), generator=gen), torch.full((n_hub,), 5, dtype=torch.int64)])
    g.edge_index = torch.cat([g.edge_index, src_hub, dst_hub], 1)
    g.edge_type = torch.cat([g.edge_type, torch.zeros(n_hub, dtype=torch.int64),
                             torch.randint(0, 3, (n_hub,), generator=gen)])
    g.edge_time = torch.cat([g.edge_time, torch.full((n_hub,), 9, dtype=torch.int64),
                             torch.randint(0, 240, (n_hub,), generator=gen)])
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
    args = (g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev), g.edge_time.to(dev))
    runs = []
    with tile_thresholds(50, 8), deterministic():
        assert 3 * P.TILE_SPLIT_EDGES <= n_hub
        for _ in range(2):
            P.clear_plan_cache()
            runs.append(_grads(m, x.to(dev), args, w.to(dev)))
        plan = P.get_plan(*args[:3], args[3], 2, 3)
        _, _, src_ix, rte_ix = P.det_index(plan, True)
        assert plan.n_hubs >= 1
        for ix in (src_ix, rte_ix):
            assert int(ix.tensors[4][2]) >= 1                   # device hub count of the source-major indices
    _assert_bitwise(runs, "hub graph")
    got = runs[0]
    for k, exp in [("<input>", xr.grad)] + [(k, params[k].grad) for k in got if k != "<input>"]:
        if exp is None:
            continue
        scale = max(exp.abs().max().item(), 1e-6)
        assert torch.allclose(got[k].cpu(), exp, rtol=2e-3, atol=2e-3 * scale), \
            "%s: max abs err %.3g (scale %.3g)" % (k, (got[k].cpu() - exp).abs().max().item(), scale)


@pytest.mark.parametrize("name", ["c1_rte", "rand_t3r4_dk4", "dense_hgt", "gnn_2layer"])
def test_deterministic_gradients_match_reference_autograd(name):
    dev = _dev()
    m, x, args, w, fx = _case(name, dev)
    with deterministic():
        P.clear_plan_cache()
        g = _grads(m, x, args, w)
    key = "grad_node_feature" if name == "gnn_2layer" else "grad_node_inp"
    _check_ref(g["<input>"], fx[key], name + " d input")
    for k, ref in fx["grad_params"].items():
        assert k in g, "no gradient for %s" % k
        _check_ref(g[k], ref, name + " d " + k)


@pytest.mark.parametrize("shape", ["mag_d256", "c3_d400"])
def test_deterministic_gradients_match_default_path(shape):
    """Flag on and off differ only in the order of floating-point sums."""
    dev = _dev()
    if shape == "mag_d256":
        g = synth.make_mag_shaped(0.01)
        d, H, rte = 256, 8, False
    else:
        g = synth.make_oag_shaped(n_nodes=20_000, n_edges=300_000)
        d, H, rte = 400, 8, True
    torch.manual_seed(0)
    m = pyhgt_b200.HGTConv(d, d, g.num_types, g.num_relations, H, 0.0, True, rte).to(dev).eval()
    x = torch.randn(g.num_nodes, d, generator=torch.Generator().manual_seed(1)).to(dev)
    w = torch.randn(g.num_nodes, d, generator=torch.Generator().manual_seed(2)).to(dev)
    args = (g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev), g.edge_time.to(dev))
    res = {}
    for on in (False, True):
        with deterministic(on):
            P.clear_plan_cache()
            res[on] = _grads(m, x, args, w)
    P.clear_plan_cache()
    bad = {k: _rel_fro(res[True][k], res[False][k]) for k in res[False]}
    bad = {k: v for k, v in bad.items() if not v <= 1e-5}
    assert not bad, bad


# ---- the edge kernels alone, through the C ABI ----------------------------------------------------------------------------

def _edge_graph(n_nodes, n_edges, T, R, seed, hubs):
    g = synth.make_random(n_nodes, n_edges, T, R, seed=seed, isolated_frac=0.1, self_loops=20, duplicate_edges=30)
    if n_edges == 0:
        empty = torch.zeros(0, dtype=torch.int64)
        return g.node_type, torch.zeros(2, 0, dtype=torch.int64), empty, empty
    ei, et, tm = g.edge_index, g.edge_type.clone(), g.edge_time
    et[::17] = R                                                 # relation out of range: these edges match no triple
    if hubs:
        gen = torch.Generator().manual_seed(seed + 1)
        k = 200
        ei = torch.cat([ei, torch.stack([torch.full((k,), 3, dtype=torch.int64), torch.randint(0, n_nodes, (k,), generator=gen)]),
                        torch.stack([torch.randint(0, n_nodes, (k,), generator=gen), torch.full((k,), 4, dtype=torch.int64)])], 1)
        et = torch.cat([et, torch.zeros(2 * k, dtype=torch.int64)])
        tm = torch.cat([tm, torch.full((2 * k,), 11, dtype=torch.int64)])
    return g.node_type, ei, et, tm


def _edge_reference(q, kv, kvr, row_ptr, kv_row, rte_row, dagg, H):
    """float64 autograd of agg_i = sum_e softmax_i(<q_i, k_e>) v_e per head; returns dq, dkv, dkvr."""
    N, d = q.shape
    dk = d // H
    q64 = q.double().requires_grad_(True)
    kv64 = kv.double().requires_grad_(True)
    kvr64 = kvr.double().requires_grad_(True) if kvr is not None else None
    deg = (row_ptr[1:] - row_ptr[:-1]).long()
    dst = torch.repeat_interleave(torch.arange(N), deg)
    k = kv64[kv_row.long(), :d]
    v = kv64[kv_row.long(), d:]
    if kvr64 is not None:
        k = k + kvr64[rte_row.long(), :d]
        v = v + kvr64[rte_row.long(), d:]
    E = dst.numel()
    s = (q64[dst].view(E, H, dk) * k.view(E, H, dk)).sum(-1)
    smax = torch.full((N, H), -float("inf"), dtype=torch.float64).scatter_reduce(
        0, dst[:, None].expand(E, H), s.detach(), "amax")
    p = torch.exp(s - smax[dst])
    den = torch.zeros(N, H, dtype=torch.float64).index_add(0, dst, p)
    p = p / (den[dst] + 1e-16)
    agg = torch.zeros(N, H, dk, dtype=torch.float64).index_add(0, dst, p[..., None] * v.view(E, H, dk))
    (agg.view(N, d) * dagg.double()).sum().backward()
    return q64.grad, kv64.grad, None if kvr64 is None else kvr64.grad


@pytest.mark.parametrize("d,H", [(32, 8), (100, 4), (256, 8), (100, 2)])    # d_k = 4, 25, 32, 50
@pytest.mark.parametrize("rte", [False, True])
@pytest.mark.parametrize("n_edges,hubs", [(3000, True), (0, False)])
def test_edge_backward_det_matches_fp64(d, H, rte, n_edges, hubs):
    dev = _dev()
    T, R, N = 3, 2, 400
    nt, ei, et, tm = _edge_graph(N, n_edges, T, R, seed=d + H, hubs=hubs)
    with tile_thresholds(37, 8):
        plan = P.get_plan(nt.to(dev), ei.to(dev), et.to(dev), tm.to(dev) if rte else None, T, R, use_cache=False)
        N, E = plan.n_nodes, plan.n_edges
        gen = torch.Generator().manual_seed(5)
        q = torch.randn(N, d, generator=gen).to(dev)
        kv = torch.randn(plan.kv_rows + 1, 2 * d, generator=gen)
        kv[-1] = 0
        kv = kv.to(dev)
        kvr = None
        if rte:
            kvr = torch.randn(plan.n_pairs * P.RTE_MAX_LEN + 1, 2 * d, generator=gen) * 0.5
            kvr[-1] = 0
            kvr = kvr.to(dev)
        dagg = torch.randn(N, d, generator=gen).to(dev)
        wsb = ctypes.c_size_t()
        _lib.call("hgt_edge_workspace_bytes", plan.n_split, d, H, ctypes.byref(wsb))
        ws = torch.empty(max(wsb.value, 1), dtype=torch.uint8, device=dev)
        agg = torch.empty(N, d, device=dev)
        stats = torch.empty(N, 2 * H, device=dev)
        _lib.call("hgt_edge_forward", q.data_ptr(), kv.data_ptr(), _lib.ptr(kvr), plan.row_ptr.data_ptr(),
                  plan.kv_row.data_ptr(), plan.rte_row.data_ptr() if rte else None, plan.csr_eid.data_ptr(),
                  plan.tiles.data_ptr(), plan.n_tiles, plan.n_split, plan.hubs.data_ptr(), plan.n_hubs, N, E, d, H, 0,
                  agg.data_ptr(), None, stats.data_ptr(), None, None, ws.data_ptr(), ws.numel(), 1,
                  _lib.ptr(plan.tile_counts_dev), plan.type_row0_dev.data_ptr(), plan.num_types, None, _stream())
        csr_dst, dst, src, rix = P.det_index(plan, rte)
        if hubs:
            assert plan.n_hubs >= 1 and int(src.tensors[4][2]) >= 1 and (not rte or int(rix.tensors[4][2]) >= 1)
        outs = []
        for _ in range(2):
            dq = torch.full((N, d), float("nan"), device=dev)
            dkv = torch.full_like(kv, float("nan"))
            dkvr = torch.full_like(kvr, float("nan")) if rte else None
            _lib.call("hgt_edge_backward_det_workspace_bytes", N, d, H, ctypes.byref(dst.c), ctypes.byref(src.c),
                      ctypes.byref(rix.c) if rte else None, ctypes.byref(wsb))
            ws2 = torch.full((wsb.value,), 255, dtype=torch.uint8, device=dev)       # NaN-patterned scratch
            _lib.call("hgt_edge_backward_det", q.data_ptr(), kv.data_ptr(), _lib.ptr(kvr), agg.data_ptr(),
                      dagg.data_ptr(), stats.data_ptr(), plan.kv_row.data_ptr(),
                      plan.rte_row.data_ptr() if rte else None, csr_dst.data_ptr(), ctypes.byref(dst.c),
                      ctypes.byref(src.c), ctypes.byref(rix.c) if rte else None, N, d, H, dq.data_ptr(), dkv.data_ptr(),
                      _lib.ptr(dkvr), ws2.data_ptr(), ws2.numel(), _stream())
            torch.cuda.synchronize()
            outs.append((dq, dkv, dkvr))
    (dq, dkv, dkvr), (dq2, dkv2, dkvr2) = outs
    assert torch.equal(dq.view(torch.int32), dq2.view(torch.int32)) and torch.equal(dkv.view(torch.int32), dkv2.view(torch.int32))
    assert E == n_edges + (20 + 30 + (400 if hubs else 0) if n_edges else 0)
    kv_row, rte_row = plan.kv_row[:E].cpu(), plan.rte_row[:E].cpu() if rte else None
    ref_dq, ref_dkv, ref_dkvr = _edge_reference(q.cpu(), kv.cpu(), None if kvr is None else kvr.cpu(),
                                                plan.row_ptr.cpu(), kv_row, rte_row, dagg.cpu(), H)
    for got, ref, what in [(dq, ref_dq, "dq"), (dkv, ref_dkv, "dkv")] + ([(dkvr, ref_dkvr, "dkvr")] if rte else []):
        assert torch.isfinite(got).all(), what + " has unwritten (NaN) entries"
        if ref.norm() > 0:
            assert _rel_fro(got, ref) <= 5e-5, "%s: rel fro %.3g" % (what, _rel_fro(got, ref))
        else:
            assert (got == 0).all(), what
    used = torch.bincount(kv_row.long(), minlength=plan.kv_rows + 1) if E else torch.zeros(plan.kv_rows + 1, dtype=torch.long)
    idle = (used == 0).nonzero().flatten()
    assert (dkv.cpu()[idle] == 0).all()                           # KV rows without out-edges: exactly zero
    if E:
        assert used[-1] > 0                                       # some edges matched no triple (the trailing row)


# ---- which kernels run -------------------------------------------------------------------------------------------------

ATOMIC_BWD_KERNELS = {"k_edge_bwd", "k_lin_dw_tc", "k_split_colsum", "k_lin_dx_simt", "k_lin_dw_simt", "k_update_bwd",
                      "k_fold_bwd_w", "k_fold_bwd_rel"}


def _step_kernels(det):
    from torch.profiler import profile, ProfilerActivity
    dev = _dev()
    g = synth.make_mag_shaped(0.01)
    torch.manual_seed(0)
    m = pyhgt_b200.HGTConv(256, 256, 4, 4, 8, 0.0, True, True).to(dev).train()      # RTE: SIMT linears too
    x = torch.randn(g.num_nodes, 256, device=dev, requires_grad=True)
    args = (g.node_type.to(dev), g.edge_index.to(dev), g.edge_type.to(dev), g.edge_time.to(dev))
    old = pyhgt_b200.HGTConv.keep_att
    pyhgt_b200.HGTConv.keep_att = False
    try:
        with deterministic(det):
            m(x, *args).sum().backward()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                m(x, *args).square().sum().backward()
                torch.cuda.synchronize()
    finally:
        pyhgt_b200.HGTConv.keep_att = old
        P.clear_plan_cache()
    names = set()
    for e in prof.key_averages():
        hit = re.search(r"\b(k_[A-Za-z0-9_]+)", e.key)
        if hit:
            names.add(hit.group(1))
    return names


def test_deterministic_step_launches_no_atomic_backward_kernel():
    names = _step_kernels(True)
    assert not names & ATOMIC_BWD_KERNELS, sorted(names & ATOMIC_BWD_KERNELS)
    for must in ("k_det_edge_dst", "k_det_edge_src", "k_det_lin_dw_tc", "k_det_split_colsum", "k_det_lin_dx_simt",
                 "k_det_lin_dw_simt", "k_det_update_bwd", "k_det_fold_w", "k_det_fold_rel", "k_ordered_sum"):
        assert must in names, (must, sorted(names))


def test_default_step_launches_no_deterministic_kernel():
    names = _step_kernels(False)
    assert not {n for n in names if n.startswith("k_det_") or n == "k_ordered_sum"}, sorted(names)
    assert {"k_edge_bwd", "k_lin_dw_tc", "k_update_bwd", "k_fold_bwd_w", "k_fold_bwd_rel"} <= names, sorted(names)


def test_sampled_batch_trains_under_the_flag_without_host_sync():
    from pyhgt_b200 import data as hdata
    from tests.test_data_ingest import _GraphStub
    dev = _dev()
    fx = load_golden("to_torch")
    g = _GraphStub(fx["types"], fx["meta_graph"])
    T = len(fx["types"])
    d = fx["node_feature"].shape[1]

    def batch():
        # edge_time stays referenced: the prebuilt plan is cached under all four tensors
        nf, nt, etime, ei, et, _, edge_dict = hdata.to_torch(fx["feature"], fx["time"], fx["edge_list"], g, device=dev,
                                                             prebuild_plan=True)
        return nf, nt, ei, et, etime, len(edge_dict)

    nf, nt, ei, et, etime, R = batch()
    torch.manual_seed(0)
    m = pyhgt_b200.HGTConv(d, d, T, R, 1, 0.0, True, False).to(dev).train()
    with deterministic():
        m(nf, nt, ei, et).sum().backward()                      # warm-up (library load, kernel attributes)
        torch.cuda.synchronize()
        P.clear_plan_cache()
        m.zero_grad(set_to_none=True)
        torch.cuda.set_sync_debug_mode("error")
        try:
            nf2, nt2, ei2, et2, etime2, _ = batch()
            m(nf2, nt2, ei2, et2).sum().backward()
        finally:
            torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    P.clear_plan_cache()
    for k, p in m.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), k
