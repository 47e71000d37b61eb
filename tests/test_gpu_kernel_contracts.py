"""GPU tests of contracts shared between kernels (run on the B200 box: ``pytest -m gpu``).

The bf16 hi/lo split: every tcgen05 GEMM takes its fp32 operands as x = hi + lo with hi = rn_bf16(x) and
lo = rn_bf16(x - hi).  Several kernels produce that split for a later GEMM (the pre-split fast paths), and sharded runs
are bit-identical to single-GPU runs only if they all round exactly alike.  Each producer's hi/lo is compared bit for
bit with the same split computed by torch."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

from pyhgt_b200 import _lib, plan as P          # noqa: E402
from tests.conftest import load_golden          # noqa: E402


def _dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _split_ref(x):
    hi = x.float().cpu().bfloat16()
    lo = (x.float().cpu() - hi.float()).bfloat16()
    return hi, lo


def _assert_split(hi, lo, x, what):
    """hi / lo (bf16, any device) must be the torch split of the fp32 tensor x, bit for bit."""
    ref_hi, ref_lo = _split_ref(x)
    x = x.cpu().flatten()
    for got, ref, part in ((hi, ref_hi, "hi"), (lo, ref_lo, "lo")):
        bad = (got.cpu().flatten().view(torch.int16) != ref.flatten().view(torch.int16)).nonzero().flatten()
        assert bad.numel() == 0, "%s: %s differs in %d of %d elements, first at x = %r" % (
            what, part, bad.numel(), x.numel(), x[bad[0]].item())


def _f32_from_bits(bits):
    """int64 tensor of 32-bit patterns -> float32."""
    return torch.where(bits >= 2**31, bits - 2**32, bits).to(torch.int32).view(torch.float32)


def _special(rows, width, seed):
    """fp32 [rows, width]: normal values over 12 decades, values exactly halfway between two bf16 numbers (ties),
    subnormals, large magnitudes (up to 1.7e38) and zeros, about half of everything negative."""
    g = torch.Generator().manual_seed(seed)
    n = rows * width
    sign = torch.randint(0, 2, (n,), generator=g) << 31
    mant = torch.randint(0, 2**23, (n,), generator=g)
    kind = torch.randint(0, 4, (n,), generator=g)
    normal = torch.randn(n, generator=g).abs() * torch.pow(10.0, torch.randint(-6, 7, (n,), generator=g).float())
    tie = (torch.randint(100, 151, (n,), generator=g) << 23) | (mant & 0x7F0000) | 0x8000
    subnormal = mant
    big = (torch.randint(0xF8, 0xFE, (n,), generator=g) << 23) | mant
    bits = torch.where(kind == 1, tie, torch.where(kind == 2, subnormal, big))
    x = torch.where(kind == 0, normal, _f32_from_bits(bits))
    x = torch.where(sign != 0, -x, x)
    x[:4] = torch.tensor([0.0, -0.0, 1.0 + 2.0**-8, -(1.0 + 3 * 2.0**-8)])     # ties rounding down and up
    return x.view(rows, width).contiguous()


def test_special_input_covers_the_cases():
    x = _special(300, 64, 1)
    b = x.view(torch.int32)
    assert ((b & 0xFFFF) == 0x8000).sum() > 1000
    assert ((x != 0) & (x.abs() < 1.17549435e-38)).sum() > 1000
    assert (x.abs() > 1e36).sum() > 1000 and (x < 0).sum() > 5000 and torch.isfinite(x).all()


@pytest.mark.parametrize("act", [0, 1])
def test_act_split_rounds_like_torch(act):
    dev = _dev()
    rows, K = 300, 64
    x = _special(rows, K, 2).to(dev)
    f32 = torch.empty_like(x)
    hi = torch.empty((rows, K), dtype=torch.bfloat16, device=dev)
    lo = torch.empty_like(hi)
    _lib.call("hgt_act_split", x.data_ptr(), K, rows, K, act, f32.data_ptr(), hi.data_ptr(), lo.data_ptr(), _stream())
    torch.cuda.synchronize()
    if act == 0:
        assert torch.equal(f32.view(torch.int32), x.view(torch.int32))
    _assert_split(hi, lo, f32, "hgt_act_split act=%d" % act)


def test_edge_forward_split_output_rounds_like_torch(monkeypatch):
    """The edge kernel writes gelu(agg) split for the a_linear GEMM; hub destinations are finished by k_merge_partials,
    which writes the split too."""
    dev = _dev()
    fx = load_golden("hub_h2")
    monkeypatch.setattr(P, "TILE_SPLIT_EDGES", 37)
    monkeypatch.setattr(P, "TILE_TARGET_EDGES", 8)
    P.clear_plan_cache()
    try:
        c = fx["cfg"]
        plan = P.get_plan(fx["node_type"].to(dev), fx["edge_index"].to(dev), fx["edge_type"].to(dev), None,
                          c["num_types"], c["num_relations"], use_cache=False)
        assert plan.n_hubs >= 1
        N, d, H = plan.n_nodes, c["out_dim"], c["n_heads"]
        g = torch.Generator().manual_seed(3)
        q = torch.randn(N, d, generator=g).to(dev)
        kv = torch.randn(plan.kv_rows + 1, 2 * d, generator=g).mul_(4.0).to(dev)
        ws_bytes = ctypes.c_size_t()
        _lib.call("hgt_edge_workspace_bytes", plan.n_split, d, H, ctypes.byref(ws_bytes))
        for variant in (1, 2):
            ws = torch.empty(max(ws_bytes.value, 1), dtype=torch.uint8, device=dev)
            agg = torch.empty(N, d, device=dev)
            hi = torch.empty(N, d, dtype=torch.bfloat16, device=dev)
            lo = torch.empty_like(hi)
            _lib.call("hgt_edge_forward", q.data_ptr(), kv.data_ptr(), None, plan.row_ptr.data_ptr(),
                      plan.kv_row.data_ptr(), None, plan.csr_eid.data_ptr(), plan.tiles.data_ptr(), plan.n_tiles,
                      plan.n_split, plan.hubs.data_ptr(), plan.n_hubs, N, plan.n_edges, d, H, 1, agg.data_ptr(), None,
                      None, hi.data_ptr(), lo.data_ptr(), ws.data_ptr(), ws.numel(), variant,
                      _lib.ptr(plan.tile_counts_dev), plan.type_row0_dev.data_ptr(), plan.num_types, None, _stream())
            torch.cuda.synchronize()
            assert agg.abs().sum() > 0
            _assert_split(hi, lo, agg, "hgt_edge_forward variant %d" % variant)
    finally:
        P.clear_plan_cache()


def test_update_epilogue_split_output_rounds_like_torch():
    dev = _dev()
    N, d = 300, 64
    x = _special(N, d, 4).to(dev)
    o = torch.zeros_like(x)
    type_row0 = torch.tensor([0, N, N], dtype=torch.int32, device=dev)
    out = torch.empty_like(x)
    hi = torch.empty(N, d, dtype=torch.bfloat16, device=dev)
    lo = torch.empty_like(hi)
    _lib.call("hgt_update_epilogue", o.data_ptr(), x.data_ptr(), type_row0.data_ptr(), 1, None, None, None, None, None,
              N, d, out.data_ptr(), hi.data_ptr(), lo.data_ptr(), _stream())
    torch.cuda.synchronize()
    assert torch.equal(out, x)                                  # y = o + x with o = 0 (+0 and -0 compare equal)
    _assert_split(hi, lo, out, "hgt_update_epilogue")


@pytest.mark.parametrize("width", [64, 256, 512, 1024])      # 1, 2, 4 and 8 float4 per lane and row
def test_halo_split_exchange_rounds_like_torch(width):
    """Single rank: the peer array holds one pointer, to this GPU's own buffer."""
    dev = _dev()
    n = 300
    x = _special(n, width, 5).to(dev)
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(6)).to(torch.int32).to(dev)
    ref = x[rows.long()]

    peers = torch.tensor([x.data_ptr()], dtype=torch.int64, device=dev)
    zeros = torch.zeros(n, dtype=torch.int32, device=dev)
    f32 = torch.empty_like(x)
    hi = torch.empty(n, width, dtype=torch.bfloat16, device=dev)
    lo = torch.empty_like(hi)
    _lib.call("hgt_halo_pull_split", peers.data_ptr(), zeros.data_ptr(), rows.data_ptr(), None, n, width, 0, 0,
              f32.data_ptr(), hi.data_ptr(), lo.data_ptr(), _stream())
    torch.cuda.synchronize()
    assert torch.equal(f32.view(torch.int32), ref.view(torch.int32))
    _assert_split(hi, lo, ref, "hgt_halo_pull_split width %d" % width)

    dst = torch.arange(n, dtype=torch.int32, device=dev)
    hi_p = torch.empty(n, width, dtype=torch.bfloat16, device=dev)
    lo_p = torch.empty_like(hi_p)
    hi_ptrs = torch.tensor([hi_p.data_ptr()], dtype=torch.int64, device=dev)
    lo_ptrs = torch.tensor([lo_p.data_ptr()], dtype=torch.int64, device=dev)
    f32_p = torch.empty_like(x)
    _lib.call("hgt_halo_push_split", x.data_ptr(), zeros.data_ptr(), rows.data_ptr(), dst.data_ptr(), n, width, 0, 0,
              hi_ptrs.data_ptr(), lo_ptrs.data_ptr(), f32_p.data_ptr(), _stream())
    torch.cuda.synchronize()
    assert torch.equal(f32_p.view(torch.int32), ref.view(torch.int32))
    _assert_split(hi_p, lo_p, ref, "hgt_halo_push_split width %d" % width)
