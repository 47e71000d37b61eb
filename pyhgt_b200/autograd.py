"""Training path of pyhgt_b200.HGTConv (reference: the same forward differentiated by autograd,
OAG/train_paper_field.py:249 ``loss.backward()``).

Every stage is a custom autograd.Function whose forward AND backward are hand-written kernels behind the C ABI:

    _FoldWeights     hgt_fold_weights / hgt_fold_backward        relation_att/msg/pri folded into the typed K/V weights
    _TypedLinear     hgt_act_split + hgt_typed_linear_presplit   typed projections, a_linears, RTE tables (tcgen05
                     / hgt_typed_linear_bwd                      split-bf16 forward, dX and dW; fp32 SIMT for odd shapes);
                                                                 the gelu in front of the a_linears (conv.py:119) lives in
                                                                 the operand split (forward) and the dX epilogue (backward)
    _EdgeAttention   hgt_edge_forward / hgt_edge_backward        score -> softmax by destination -> weighted aggregation
    _UpdateEpilogue  hgt_update_epilogue / hgt_update_backward   sigmoid(skip) gate + LayerNorm (conv.py:129-133)

Under ``torch.use_deterministic_algorithms(True)`` (read when a backward runs, like PyTorch's own ops) every backward
stage takes its ``*_det`` entry point instead: the same gradients up to summation order, with every sum in an order fixed
by the problem shape (no floating-point atomics), so the gradient bits repeat from run to run.  The edge backward then
runs source-major over an index built on first use and cached on the plan (plan.det_index).

No per-edge intermediates are kept: the edge backward recomputes the softmax weights from the saved per-destination
(max, sum); the typed linears keep the bf16 hi/lo split of their input (the A operand of the dW product).  No cuBLAS,
no torch matmul on this path.  Gradients reach ``node_inp`` and every parameter of conv.py:28-54 including ``emb.*``.
The inference path (``torch.no_grad``) does not come through here: it uses the fused kernels in conv.py.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from . import plan as _plan


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _det():
    return torch.are_deterministic_algorithms_enabled()


def _det_scratch(nbytes, dev):
    """Workspace of a *_det call.  Those calls write every scratch byte before reading it, so the NaN fill torch gives
    torch.empty under deterministic mode (fill_uninitialized_memory) would only cost a pass over it."""
    det_mod = torch.utils.deterministic
    fill = det_mod.fill_uninitialized_memory
    det_mod.fill_uninitialized_memory = False
    try:
        return torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
    finally:
        det_mod.fill_uninitialized_memory = fill


def _tc_shape_ok(K, width):
    """Shapes both the tensor-core forward (hgt_typed_linear_presplit) and backward (hgt_typed_linear_bwd) take."""
    return K % 16 == 0 and K >= 64 and width % 16 == 0


class _TypedLinear(torch.autograd.Function):
    """out_flat[cblock c of group g][m, :] = act(A)[rows_g] @ W_cat[rows of (g, c)]^T + b_cat   (act: 0 none, 1 gelu)."""

    @staticmethod
    def forward(ctx, a, w_cat, b_cat, table, width, out_elems, impl, act, zero_ranges):
        g_dev, g_host, n_g, c_dev = table
        a = a.contiguous()
        w_cat = w_cat.contiguous()
        rows, K = a.shape
        dev = a.device
        st = _stream()
        out = torch.empty(out_elems, dtype=torch.float32, device=dev)
        for (z0, z1) in zero_ranges:                                   # padding / all-zero table rows only
            if z1 > z0:
                out[z0:z1].zero_()
        use_tc = impl in (0, 2) and _tc_shape_ok(K, width)
        hi = lo = a_act = None
        wsb = ctypes.c_size_t()
        if use_tc:
            hi = torch.empty((rows, K), dtype=torch.bfloat16, device=dev)
            lo = torch.empty((rows, K), dtype=torch.bfloat16, device=dev)
            _lib.call("hgt_act_split", a.data_ptr(), K, rows, K, act, None, hi.data_ptr(), lo.data_ptr(), st)
            _lib.call("hgt_typed_linear_presplit_workspace_bytes", g_host.ctypes.data, n_g, K, width, ctypes.byref(wsb))
            ws = torch.empty(max(wsb.value, 1), dtype=torch.uint8, device=dev)
            _lib.call("hgt_typed_linear_presplit", hi.data_ptr(), lo.data_ptr(), w_cat.data_ptr(), _lib.ptr(b_cat), K, width,
                      g_dev.data_ptr(), g_host.ctypes.data, n_g, c_dev.data_ptr(), out.data_ptr(), ws.data_ptr(),
                      ws.numel(), st)
        else:
            a_act = a
            if act:
                a_act = torch.empty_like(a)
                _lib.call("hgt_act_split", a.data_ptr(), K, rows, K, act, a_act.data_ptr(), None, None, st)
            _lib.call("hgt_typed_linear_workspace_bytes", g_host.ctypes.data, n_g, K, width, 1, ctypes.byref(wsb))
            ws = torch.empty(max(wsb.value, 1), dtype=torch.uint8, device=dev)
            _lib.call("hgt_typed_linear", a_act.data_ptr(), K, w_cat.data_ptr(), _lib.ptr(b_cat), K, width,
                      g_dev.data_ptr(), g_host.ctypes.data, n_g, c_dev.data_ptr(), out.data_ptr(), 1, ws.data_ptr(),
                      ws.numel(), st)
        ctx.table, ctx.width, ctx.has_bias, ctx.act, ctx.use_tc = table, width, b_cat is not None, act, use_tc
        ctx.out_elems = out_elems
        # gelu'(a) needs the un-activated input; the dW product needs act(a): as the bf16 split (tensor cores) or fp32
        ctx.save_for_backward(a if (act or not use_tc) else None, a_act if (act and not use_tc) else None, hi, lo, w_cat)
        return out

    @staticmethod
    def backward(ctx, dout):
        a, a_act, hi, lo, w_cat = ctx.saved_tensors
        width = ctx.width
        K = w_cat.shape[1]
        dev = w_cat.device
        rows = hi.shape[0] if hi is not None else a.shape[0]
        need_da = ctx.needs_input_grad[0]
        dout = dout.contiguous()
        da = torch.empty((rows, K), dtype=torch.float32, device=dev) if need_da else None
        dw = torch.zeros_like(w_cat)                                   # small: [sum of out rows, K]
        db = torch.zeros(w_cat.shape[0], dtype=torch.float32, device=dev) if ctx.has_bias else None
        impl = 2 if ctx.use_tc else 1
        fn = "hgt_typed_linear_bwd_det" if _det() else "hgt_typed_linear_bwd"
        a_f32 = a_act if a_act is not None else a                      # SIMT dW operand (act already applied)
        # tables whose groups overlap in rows (sharded per-pair compaction) come with disjoint sub-tables: the first call
        # writes dA, the others accumulate into it; dW / db accumulate anyway
        tables = getattr(ctx.table, "bwd_tables", None) or [ctx.table]
        if not ctx.use_tc:
            tables = [ctx.table]                                       # the SIMT dX adds up overlapping groups itself
        if need_da:
            # hgt_typed_linear_bwd zeroes the gaps between the first table's groups; rows past its last group (other
            # sub-tables' rows, nodes of unknown type) are zeroed here
            g0, n0 = tables[0][1], tables[0][2]
            end0 = int((g0["a_row0"][:n0] + g0["m"][:n0]).max()) if n0 else 0
            if end0 < rows:
                da[end0:].zero_()
        for ti, tab in enumerate(tables):
            g_dev, g_host, n_g, _ = tab
            c_host = tab.c_host
            wsb = ctypes.c_size_t()
            _lib.call(fn + "_workspace_bytes", g_host.ctypes.data, n_g, c_host.ctypes.data, K, width, K,
                      ctx.out_elems, 0, int(hi is not None), impl, ctypes.byref(wsb))
            ws = (_det_scratch(wsb.value, dev) if fn.endswith("_det") else
                  torch.empty(max(wsb.value, 1), dtype=torch.uint8, device=dev))
            _lib.call(fn, dout.data_ptr(), None, None, ctx.out_elems, _lib.ptr(a_f32), K, _lib.ptr(hi),
                      _lib.ptr(lo), w_cat.data_ptr(), K, width, g_dev.data_ptr(), g_host.ctypes.data, n_g,
                      c_host.ctypes.data, _lib.ptr(da), int(ti > 0), a.data_ptr() if ctx.act else None, dw.data_ptr(),
                      _lib.ptr(db), impl, ws.data_ptr(), ws.numel(), _stream())
        return da, dw, db, None, None, None, None, None, None


class _EdgeAttention(torch.autograd.Function):
    """agg[i] = sum_{e -> i} softmax_i(<Q[i], K'[e]>) * V'[e]   (conv.py:99,108-111 + scatter-add).  Takes and returns
    the FLAT projection buffer (Q at q_off, the [K'|V'] table at kv_off): its gradient is produced as one buffer, so
    autograd never assembles it from slices."""

    @staticmethod
    def forward(ctx, proj, kvr, plan, lt, d, n_heads, want_att, variant):
        N = plan.n_nodes
        dev = proj.device
        proj = proj.contiguous()
        q = proj[lt.q_off:lt.q_off + N * d]
        kv = proj[lt.kv_off:]
        ws_bytes = ctypes.c_size_t()
        _lib.call("hgt_edge_workspace_bytes", plan.n_split, d, n_heads, ctypes.byref(ws_bytes))
        ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=dev)
        agg = torch.empty((N, d), dtype=torch.float32, device=dev)
        stats = torch.empty((N, 2 * n_heads), dtype=torch.float32, device=dev)
        att = torch.empty((plan.n_edges, n_heads), dtype=torch.float32, device=dev) if want_att else None
        kvr = None if kvr is None else kvr.contiguous()
        _lib.call("hgt_edge_forward", q.data_ptr(), kv.data_ptr(), _lib.ptr(kvr), plan.row_ptr.data_ptr(),
                  plan.kv_row.data_ptr(), None if kvr is None else plan.rte_row.data_ptr(), plan.csr_eid.data_ptr(),
                  plan.tiles.data_ptr(), plan.n_tiles, plan.n_split, plan.hubs.data_ptr(), plan.n_hubs, N, plan.n_edges, d,
                  n_heads, 0, agg.data_ptr(), _lib.ptr(att), stats.data_ptr(), None, None, ws.data_ptr(), ws.numel(),
                  variant, _lib.ptr(plan.tile_counts_dev), plan.type_row0_dev.data_ptr(), plan.num_types,
                  _lib.ptr(lt.type_active_dev), _stream())
        ctx.plan, ctx.lt, ctx.d, ctx.n_heads, ctx.has_kvr = plan, lt, d, n_heads, kvr is not None
        ctx.save_for_backward(proj, kvr, agg, stats)
        if att is not None:
            ctx.mark_non_differentiable(att)
        return agg, att

    @staticmethod
    def backward(ctx, dagg, _datt=None):
        proj, kvr, agg, stats = ctx.saved_tensors
        plan, lt, d, H = ctx.plan, ctx.lt, ctx.d, ctx.n_heads
        N = plan.n_nodes
        q = proj[lt.q_off:lt.q_off + N * d]
        kv = proj[lt.kv_off:]
        dproj = torch.empty_like(proj)                                 # hgt_edge_backward zero-initialises dq / dkv
        if lt.kv_off > N * d:
            dproj[N * d:lt.kv_off].zero_()                             # alignment gap
        dq = dproj[lt.q_off:lt.q_off + N * d]
        dkv = dproj[lt.kv_off:]
        dkvr = torch.empty_like(kvr) if kvr is not None else None
        dagg = dagg.contiguous()
        if _det():
            # every row of dq / dkv / dkvr is written by the call: no zero fill
            csr_dst, dst, src, rte = _plan.det_index(plan, kvr is not None)
            wsb = ctypes.c_size_t()
            _lib.call("hgt_edge_backward_det_workspace_bytes", N, d, H, ctypes.byref(dst.c), ctypes.byref(src.c),
                      None if rte is None else ctypes.byref(rte.c), ctypes.byref(wsb))
            ws = _det_scratch(wsb.value, proj.device)
            _lib.call("hgt_edge_backward_det", q.data_ptr(), kv.data_ptr(), _lib.ptr(kvr), agg.data_ptr(),
                      dagg.data_ptr(), stats.data_ptr(), plan.kv_row.data_ptr(),
                      None if kvr is None else plan.rte_row.data_ptr(), csr_dst.data_ptr(), ctypes.byref(dst.c),
                      ctypes.byref(src.c), None if rte is None else ctypes.byref(rte.c), N, d, H, dq.data_ptr(),
                      dkv.data_ptr(), _lib.ptr(dkvr), ws.data_ptr(), ws.numel(), _stream())
            return dproj, dkvr, None, None, None, None, None, None
        ws = torch.empty(256, dtype=torch.uint8, device=proj.device)
        _lib.call("hgt_edge_backward", q.data_ptr(), kv.data_ptr(), _lib.ptr(kvr), agg.data_ptr(), dagg.data_ptr(),
                  stats.data_ptr(), plan.row_ptr.data_ptr(), plan.kv_row.data_ptr(),
                  None if kvr is None else plan.rte_row.data_ptr(), plan.tiles.data_ptr(), plan.n_tiles, N, d, H,
                  plan.kv_rows + 1, 0 if kvr is None else kvr.numel() // (2 * d),
                  dq.data_ptr(), dkv.data_ptr(), _lib.ptr(dkvr), ws.data_ptr(), ws.numel(),
                  _lib.ptr(plan.tile_counts_dev), _stream())
        return dproj, dkvr, None, None, None, None, None, None


class _FoldWeights(torch.autograd.Function):
    """(W_cat, b_cat) of the typed projection: per type  [W_q ; K'_p ; V'_p ...]  (hgt_fold_weights, conv.py:96-104)."""

    @staticmethod
    def forward(ctx, module, plan, lt, *params):
        m = module
        T, R, H, d_in, d = m.num_types, m.num_relations, m.n_heads, m.in_dim, m.out_dim
        dev = params[0].device
        st = _stream()
        tabs = [m._ptrs(n, ts, dev) for n, ts in (("wq", [l.weight for l in m.q_linears]), ("bq", [l.bias for l in m.q_linears]),
                                                 ("wk", [l.weight for l in m.k_linears]), ("bk", [l.bias for l in m.k_linears]),
                                                 ("wv", [l.weight for l in m.v_linears]), ("bv", [l.bias for l in m.v_linears]))]
        w_cat = torch.empty((max(lt.cat_rows, 1), d_in), dtype=torch.float32, device=dev)
        b_cat = torch.empty(max(lt.cat_rows, 1), dtype=torch.float32, device=dev)
        _lib.call("hgt_fold_weights", *[t.data_ptr() for t in tabs], m.relation_att.data_ptr(), m.relation_msg.data_ptr(),
                  m.relation_pri.data_ptr(), T, R, H, d_in, d, plan.n_pairs, plan.pair_type_dev.data_ptr(),
                  plan.pair_rel_dev.data_ptr(), lt.cat_row0_dev.data_ptr(), lt.q_row0_dev.data_ptr(), w_cat.data_ptr(),
                  b_cat.data_ptr(), st)
        ctx.module, ctx.plan, ctx.lt, ctx.tabs = m, plan, lt, tabs
        return w_cat, b_cat

    @staticmethod
    def backward(ctx, dw_cat, db_cat):
        m, plan, lt, tabs = ctx.module, ctx.plan, ctx.lt, ctx.tabs
        T, R, H, d_in, d, dk = m.num_types, m.num_relations, m.n_heads, m.in_dim, m.out_dim, m.d_k
        dev = dw_cat.device
        dw_cat, db_cat = dw_cat.contiguous(), db_cat.contiguous()
        f32 = dict(dtype=torch.float32, device=dev)
        d_wk, d_wv = torch.empty((T, d, d_in), **f32), torch.empty((T, d, d_in), **f32)
        d_bk, d_bv = torch.empty((T, d), **f32), torch.empty((T, d), **f32)
        d_att, d_msg = torch.empty((R, H, dk, dk), **f32), torch.empty((R, H, dk, dk), **f32)
        d_pri = torch.empty((R, H), **f32)
        args = (dw_cat.data_ptr(), db_cat.data_ptr(), tabs[2].data_ptr(), tabs[3].data_ptr(),
                tabs[4].data_ptr(), tabs[5].data_ptr(), m.relation_att.data_ptr(), m.relation_msg.data_ptr(),
                m.relation_pri.data_ptr(), T, R, H, d_in, d, plan.n_pairs, plan.pair_type_dev.data_ptr(),
                plan.pair_rel_dev.data_ptr(), lt.cat_row0_dev.data_ptr(), d_wk.data_ptr(), d_bk.data_ptr(),
                d_wv.data_ptr(), d_bv.data_ptr(), d_att.data_ptr(), d_msg.data_ptr(), d_pri.data_ptr())
        if _det():
            wsb = ctypes.c_size_t()
            _lib.call("hgt_fold_backward_det_workspace_bytes", R, H, d, ctypes.byref(wsb))
            ws = _det_scratch(wsb.value, dev)
            _lib.call("hgt_fold_backward_det", *args, ws.data_ptr(), ws.numel(), _stream())
        else:
            _lib.call("hgt_fold_backward", *args, _stream())
        # W_q / b_q rows of W_cat are plain copies: their gradient is the matching slice
        d_wq = [dw_cat[lt.q_row0[t]:lt.q_row0[t] + d] for t in range(T)]
        d_bq = [db_cat[lt.q_row0[t]:lt.q_row0[t] + d] for t in range(T)]
        grads = d_wq + d_bq + list(d_wk.unbind(0)) + list(d_bk.unbind(0)) + list(d_wv.unbind(0)) + list(d_bv.unbind(0))
        return (None, None, None) + tuple(grads) + (d_att, d_msg, d_pri)


class _UpdateEpilogue(torch.autograd.Function):
    """out[perm[k]] = LayerNorm_t(o[k] * sigmoid(skip[t]) + x[k] * (1 - sigmoid(skip[t])))   (conv.py:129-133);
    skip=None: the plain residual o + x of DenseHGTConv (conv.py:261,273).  type_row0: [T+2] int32 row prefix (rows past
    type_row0[T] are written as zeros), perm: rank-order row -> output row, or None."""

    @staticmethod
    def forward(ctx, o, x, skip, norm_w, norm_b, type_row0, T, perm, type_active=None):
        N, d = o.shape
        o, x = o.contiguous(), x.contiguous()
        # with type_active (sharded training) the rows past the active prefix of a type have no output row: they stay
        # unwritten (the caller selects the owned rows) and receive no gradient (hgt_update_backward skips them)
        out = torch.empty((N, d), dtype=torch.float32, device=o.device)
        _lib.call("hgt_update_epilogue", o.data_ptr(), x.data_ptr(), type_row0.data_ptr(), T, _lib.ptr(skip),
                  _lib.ptr(norm_w), _lib.ptr(norm_b), _lib.ptr(perm), _lib.ptr(type_active), N, d, out.data_ptr(), None,
                  None, _stream())
        ctx.T, ctx.has_norm, ctx.has_skip = T, norm_w is not None, skip is not None
        ctx.save_for_backward(o, x, skip, norm_w, type_row0, perm, type_active)
        return out

    @staticmethod
    def backward(ctx, dout):
        o, x, skip, norm_w, type_row0, perm, type_active = ctx.saved_tensors
        T = ctx.T
        N, d = o.shape
        dev = o.device
        dout = dout.contiguous()
        d_o, d_x = torch.empty_like(o), torch.empty_like(x)
        d_skip = torch.empty(T, dtype=torch.float32, device=dev) if ctx.has_skip else None
        d_nw = torch.empty((T, d), dtype=torch.float32, device=dev) if ctx.has_norm else None
        d_nb = torch.empty((T, d), dtype=torch.float32, device=dev) if ctx.has_norm else None
        args = (dout.data_ptr(), o.data_ptr(), x.data_ptr(), type_row0.data_ptr(), T,
                _lib.ptr(skip), _lib.ptr(norm_w), _lib.ptr(perm), _lib.ptr(type_active), N, d, d_o.data_ptr(),
                d_x.data_ptr(), _lib.ptr(d_skip), _lib.ptr(d_nw), _lib.ptr(d_nb))
        if _det():
            wsb = ctypes.c_size_t()
            _lib.call("hgt_update_backward_det_workspace_bytes", N, T, d, ctypes.byref(wsb))
            ws = _det_scratch(wsb.value, dev)
            _lib.call("hgt_update_backward_det", *args, ws.data_ptr(), ws.numel(), _stream())
        else:
            _lib.call("hgt_update_backward", *args, _stream())
        return d_o, d_x, d_skip, d_nw, d_nb, None, None, None, None


def typed_linear(a, w_cat, b_cat, table, width, out_elems, impl=0, act=0, zero_ranges=()):
    return _TypedLinear.apply(a, w_cat, b_cat, table, width, out_elems, impl, act, tuple(zero_ranges))


def hgt_conv_autograd(m, node_inp, node_type, edge_index, edge_type, edge_time, active=None, kv_runs=None):
    """`active` (sharded training): active[t] = number of leading nodes of type t (rank order) that are destinations on
    this rank; Q / a_linear / update run for them only, the remaining rows (halo sources) only get K'/V' rows and their
    output rows stay zero.  `kv_runs`: per-pair row ranges that need K'/V' (plan.layer_tables)."""
    d_in, d, H, T, R = m.in_dim, m.out_dim, m.n_heads, m.num_types, m.num_relations
    plan = _plan.get_plan(node_type, edge_index, edge_type, edge_time if m.use_RTE else None, T, R)
    N, P = plan.n_nodes, plan.n_pairs
    if node_inp.shape[0] != N:
        raise ValueError("node_inp has %d rows but node_type has %d" % (node_inp.shape[0], N))
    x = node_inp if plan.sorted_types else node_inp.index_select(0, plan.perm.long())
    if active is not None and not plan.sorted_types:
        raise ValueError("`active` needs a type-sorted node order")
    lt = _plan.layer_tables(plan, d_in, d, active, kv_runs)

    # 1. relation matrices folded into the typed K/V weights; typed projections -> flat [Q | pad | K'V' table | zero row]
    params = ([l.weight for l in m.q_linears] + [l.bias for l in m.q_linears] +
              [l.weight for l in m.k_linears] + [l.bias for l in m.k_linears] +
              [l.weight for l in m.v_linears] + [l.bias for l in m.v_linears] +
              [m.relation_att, m.relation_msg, m.relation_pri])
    w_cat, b_cat = _FoldWeights.apply(m, plan, lt, *params)
    kv_end = lt.kv_off + plan.kv_rows * 2 * d
    proj = typed_linear(x, w_cat, b_cat, lt.proj_groups, d, lt.proj_elems, m.linear_impl, 0,
                        ((N * d, lt.kv_off), (kv_end, lt.proj_elems)))
    kvr = None
    if m.use_RTE:
        # RT = lin(emb.weight) [240, d_in] (conv.py:299), then projected with every pair's K'/V' weights (no bias)
        rt = typed_linear(m.emb.emb.weight, m.emb.lin.weight, m.emb.lin.bias, lt.rt_group, d_in,
                          _plan.RTE_MAX_LEN * d_in, 1).view(_plan.RTE_MAX_LEN, d_in)
        n_kvr = (P * _plan.RTE_MAX_LEN + 1) * 2 * d
        kvr = typed_linear(rt, w_cat, None, lt.rte_groups, d, n_kvr, 1, 0, ((P * _plan.RTE_MAX_LEN * 2 * d, n_kvr),))

    # 2. fused edge kernel
    agg, att = _EdgeAttention.apply(proj, kvr, plan, lt, d, H, bool(m.keep_att), m.edge_variant)
    m.att = att

    # 3. a_linears on gelu(agg) (conv.py:119,125): the gelu is applied inside the operand split / the dX epilogue
    wa_cat = torch.cat([l.weight for l in m.a_linears], 0)
    ba_cat = torch.cat([l.bias for l in m.a_linears], 0)
    o = typed_linear(agg, wa_cat, ba_cat, lt.upd_groups, d, N * d, m.linear_impl, 1).view(N, d)
    if m.training and m.drop.p > 0:
        o = m.drop(o)                                                            # conv.py:125

    # 4. gated skip + LayerNorm, written in original node order; rows of unknown type stay zero (conv.py:120)
    norm_w = torch.stack([n.weight for n in m.norms]) if m.use_norm else None
    norm_b = torch.stack([n.bias for n in m.norms]) if m.use_norm else None
    return _UpdateEpilogue.apply(o, x, m.skip, norm_w, norm_b, plan.type_row0_dev, T,
                                 None if plan.sorted_types else plan.perm, lt.type_active_dev)


def dense_hgt_forward(m, node_inp, node_type, edge_index, edge_type, edge_time):
    """DenseHGTConv.forward (conv.py:143-280): the same message() => the same projection / edge kernels, then
        y   = LayerNorm_t(drop(a_linear_t(agg)) + x)                     conv.py:261-266   (no gelu, no skip gate)
        out = out_norm(drop(out_linear(gelu(mid_linear(y)))) + y)        conv.py:273-274   (FFN shared by all types)
    built from the same differentiable stages: typed GEMMs (the gelu of the FFN sits in the operand split of out_linear
    and in the dX epilogue of its backward) and the residual mode of the update epilogue.  Used for inference and
    training alike (under no_grad the stages simply do not record)."""
    d_in, d, H, T, R = m.in_dim, m.out_dim, m.n_heads, m.num_types, m.num_relations
    plan = _plan.get_plan(node_type, edge_index, edge_type, edge_time if m.use_RTE else None, T, R)
    N, P = plan.n_nodes, plan.n_pairs
    if node_inp.shape[0] != N:
        raise ValueError("node_inp has %d rows but node_type has %d" % (node_inp.shape[0], N))
    dev = node_inp.device
    x = node_inp if plan.sorted_types else node_inp.index_select(0, plan.perm.long())
    lt = _plan.layer_tables(plan, d_in, d)
    params = ([l.weight for l in m.q_linears] + [l.bias for l in m.q_linears] +
              [l.weight for l in m.k_linears] + [l.bias for l in m.k_linears] +
              [l.weight for l in m.v_linears] + [l.bias for l in m.v_linears] +
              [m.relation_att, m.relation_msg, m.relation_pri])
    w_cat, b_cat = _FoldWeights.apply(m, plan, lt, *params)
    kv_end = lt.kv_off + plan.kv_rows * 2 * d
    proj = typed_linear(x, w_cat, b_cat, lt.proj_groups, d, lt.proj_elems, m.linear_impl, 0,
                        ((N * d, lt.kv_off), (kv_end, lt.proj_elems)))
    kvr = None
    if m.use_RTE:
        rt = typed_linear(m.emb.emb.weight, m.emb.lin.weight, m.emb.lin.bias, lt.rt_group, d_in,
                          _plan.RTE_MAX_LEN * d_in, 1).view(_plan.RTE_MAX_LEN, d_in)
        n_kvr = (P * _plan.RTE_MAX_LEN + 1) * 2 * d
        kvr = typed_linear(rt, w_cat, None, lt.rte_groups, d, n_kvr, 1, 0, ((P * _plan.RTE_MAX_LEN * 2 * d, n_kvr),))
    agg, att = _EdgeAttention.apply(proj, kvr, plan, lt, d, H, bool(m.keep_att), m.edge_variant)
    m.att = att

    drop = m.training and m.drop.p > 0
    wa_cat = torch.cat([l.weight for l in m.a_linears], 0)
    ba_cat = torch.cat([l.bias for l in m.a_linears], 0)
    o = typed_linear(agg, wa_cat, ba_cat, lt.upd_groups, d, N * d, m.linear_impl, 0).view(N, d)     # conv.py:261
    if drop:
        o = m.drop(o)
    norm_w = torch.stack([n.weight for n in m.norms]) if m.use_norm else None
    norm_b = torch.stack([n.bias for n in m.norms]) if m.use_norm else None
    y = _UpdateEpilogue.apply(o, x, None, norm_w, norm_b, plan.type_row0_dev, T, None)              # rank order

    n_known = plan.type_row0[T]
    key = ("dense_ffn", d)
    tabs = plan._layer_tables.get(key)
    if tabs is None:
        one = lambda w_: _plan._pack_groups([(0, n_known, 0, 1, 0, 1)], [(0, w_)], dev)            # noqa: E731
        tabs = plan._layer_tables[key] = (one(2 * d), one(d),
                                          _plan._to_dev_async(np.asarray([0, n_known, N], dtype=np.int32), dev))
    hmid = typed_linear(y, m.mid_linear.weight, m.mid_linear.bias, tabs[0], 2 * d, N * 2 * d, m.linear_impl, 0,
                        ((n_known * 2 * d, N * 2 * d),)).view(N, 2 * d)
    z = typed_linear(hmid, m.out_linear.weight, m.out_linear.bias, tabs[1], d, N * d, m.linear_impl, 1,
                     ((n_known * d, N * d),)).view(N, d)                                             # gelu inside
    if drop:
        z = m.drop(z)
    # shared out_norm over every known row, residual with y, written in original node order; unknown types -> zeros
    return _UpdateEpilogue.apply(z, y, None, m.out_norm.weight.view(1, d), m.out_norm.bias.view(1, d), tabs[2], 1,
                                 None if plan.sorted_types else plan.perm)
