"""Drop-in replacements for pyHGT's conv layer classes (reference: pyHGT/conv.py).

``HGTConv`` keeps the reference's constructor (conv.py:12), five-argument ``forward`` (conv.py:56),
public attributes (conv.py:15-25), ``.att`` side effect (conv.py:108), ``__repr__`` (conv.py:136-139) and
parameter / state_dict names (conv.py:28-54), but computes through the hand-written sm_100a kernels
behind the C ABI in include/hgt_b200.h:

    plan (once per graph)            hgt_plan_*          CSR by destination, pairs, gather rows, tiles
    fold relation matrices           hgt_fold_weights    relation_att/msg/pri -> per-<type,relation> W'
    typed projections                hgt_typed_linear    Q [N,d] and [K'|V'] tables (+ RTE tables)
    fused edge kernel                hgt_edge_forward    score -> softmax by destination -> weighted sum (+gelu)
    typed output linear              hgt_typed_linear    a_linears
    gated skip + LayerNorm           hgt_update_epilogue

``HGTConv.kv_dtype = torch.bfloat16`` (or ``set_kv_dtype``) is an opt-in inference mode: the folded [K'|V'] table and
the RTE tables K'R/V'R are stored as bf16 (each row rounded to nearest even after its fp32 GEMM), which halves the
bytes the edge kernel gathers; Q, every sum, the softmax, ``att`` and the output stay fp32.

There is no CPU path: CPU tensors raise.  ``GeneralConv`` mirrors conv.py:303-323 so that pyHGT's
model.py (``from .conv import *``) runs unchanged on top of this module.
"""
import ctypes
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from . import plan as _plan


def glorot(tensor):
    """torch_geometric.nn.inits.glorot (used at conv.py:53-54)."""
    if tensor is not None:
        a = math.sqrt(6.0 / (tensor.size(-2) + tensor.size(-1)))
        tensor.data.uniform_(-a, a)


class RelTemporalEncoding(nn.Module):
    """Sinusoid table + linear (reference conv.py:283-299).  Same parameter names (emb.weight,
    lin.weight, lin.bias).  Inside HGTConv the table is never applied per edge: RT = lin(emb.weight)
    [240,d] is projected once per <source type, relation> and added per edge by the edge kernel."""

    def __init__(self, n_hid, max_len=240, dropout=0.2):
        super().__init__()
        position = torch.arange(0., max_len).unsqueeze(1)
        div_term = torch.exp(torch.arange(0, n_hid, 2) * -(math.log(10000.0) / n_hid))
        emb = nn.Embedding(max_len, n_hid)
        emb.weight.data[:, 0::2] = torch.sin(position * div_term) / math.sqrt(n_hid)
        emb.weight.data[:, 1::2] = torch.cos(position * div_term) / math.sqrt(n_hid)
        emb.requires_grad = False        # (sic) the reference sets a module attribute: the table stays trainable
        self.emb = emb
        self.lin = nn.Linear(n_hid, n_hid)

    def forward(self, x, t):
        return x + self.lin(self.emb(t))


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _PointerTable:
    """Device array of per-type parameter pointers, rebuilt only when a parameter moves."""

    def __init__(self):
        self.key = None
        self.dev = None

    def get(self, tensors, device):
        key = tuple(t.data_ptr() for t in tensors) + (str(device),)
        if key != self.key:
            self.dev = torch.tensor([t.data_ptr() for t in tensors], dtype=torch.int64).to(device)
            self.key = key
        return self.dev


class HGTConv(nn.Module):
    # Class-level switches (kept out of the constructor so the reference's positional call at
    # conv.py:308 stays valid).
    keep_att = True            # materialise self.att [E,H] like the reference (conv.py:108)
    edge_variant = 0           # 0 auto, 1 register gather, 2 bulk-copy ring (see csrc/edge.cu)
    linear_impl = 0            # 0 auto, 1 fp32 SIMT, 2 tcgen05
    event_sink = None          # bench.py: list receiving (stage, start_event, end_event) on the launch stream
    _has_skip = True           # DenseHGTConv (conv.py:143-280) has no skip gate
    emit_split = False         # also write the output as a bf16 hi/lo split for the next layer (model.GNN sets it)
    fused_call = True          # inference goes through ONE C-ABI call (hgt_conv_forward) instead of ~12
    kv_dtype = torch.float32   # torch.bfloat16: inference with bf16 [K'|V'] / K'R/V'R tables (see set_kv_dtype)

    def __init__(self, in_dim, out_dim, num_types, num_relations, n_heads, dropout=0.2, use_norm=True,
                 use_RTE=True, **kwargs):
        super().__init__()
        self.in_dim = in_dim
        self.out_dim = out_dim
        self.num_types = num_types
        self.num_relations = num_relations
        self.total_rel = num_types * num_relations * num_types
        self.n_heads = n_heads
        self.d_k = out_dim // n_heads
        self.sqrt_dk = math.sqrt(self.d_k)
        self.use_norm = use_norm
        self.use_RTE = use_RTE
        self.att = None

        self.k_linears = nn.ModuleList()
        self.q_linears = nn.ModuleList()
        self.v_linears = nn.ModuleList()
        self.a_linears = nn.ModuleList()
        self.norms = nn.ModuleList()
        for _ in range(num_types):
            self.k_linears.append(nn.Linear(in_dim, out_dim))
            self.q_linears.append(nn.Linear(in_dim, out_dim))
            self.v_linears.append(nn.Linear(in_dim, out_dim))
            self.a_linears.append(nn.Linear(out_dim, out_dim))
            if use_norm:
                self.norms.append(nn.LayerNorm(out_dim))
        self.relation_pri = nn.Parameter(torch.ones(num_relations, self.n_heads))
        self.relation_att = nn.Parameter(torch.Tensor(num_relations, n_heads, self.d_k, self.d_k))
        self.relation_msg = nn.Parameter(torch.Tensor(num_relations, n_heads, self.d_k, self.d_k))
        if self._has_skip:
            self.skip = nn.Parameter(torch.ones(num_types))
        self.drop = nn.Dropout(dropout)
        if self.use_RTE:
            self.emb = RelTemporalEncoding(in_dim)
        glorot(self.relation_att)
        glorot(self.relation_msg)
        self._ptr_tables = {}

    def __repr__(self):
        return '{}(in_dim={}, out_dim={}, num_types={}, num_types={})'.format(
            self.__class__.__name__, self.in_dim, self.out_dim, self.num_types, self.num_relations)

    def __getstate__(self):
        """Launch caches (ctypes argument blocks, device pointer tables, pinned plans) are per-process state: they are
        dropped from the pickled / deep-copied module so `torch.save(model)` (OAG/train_paper_field.py:279) works after
        a forward; they are rebuilt lazily."""
        state = self.__dict__.copy()
        state.pop("_args_cache", None)
        state["_ptr_tables"] = {}
        return state

    # ------------------------------------------------------------------------------------------
    def _ptrs(self, name, tensors, device):
        tab = self._ptr_tables.get(name)
        if tab is None:
            tab = self._ptr_tables[name] = _PointerTable()
        return tab.get(tensors, device)

    @staticmethod
    def _stage(name):
        """Context manager recording CUDA events around a stage when HGTConv.event_sink is a list (bench.py)."""
        class _T:
            def __enter__(self_):
                self_.on = HGTConv.event_sink is not None
                if self_.on:
                    self_.a, self_.b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    self_.a.record()
            def __exit__(self_, *exc):
                if self_.on:
                    self_.b.record()
                    HGTConv.event_sink.append((name, self_.a, self_.b))
        return _T()

    def _typed_linear(self, a, lda, w, bias, k, width, table, out, impl, st, groups=None):
        """hgt_typed_linear with its (impl-dependent) workspace; table = (groups_dev, groups_host, n, cblocks_dev).
        `groups` = (first, count) restricts the call to a range of the table's groups.  A bf16 `out` selects
        hgt_typed_linear_bf16 (the same product, rounded to bf16 as it is stored)."""
        g_dev, g_host, n_g, c_dev = table
        first, n_g = (0, n_g) if groups is None else groups
        g_ptr, h_ptr = g_dev.data_ptr() + first * g_host.itemsize, g_host.ctypes.data + first * g_host.itemsize
        sfx = "_bf16" if out.dtype == torch.bfloat16 else ""
        ws_bytes = ctypes.c_size_t()
        _lib.call("hgt_typed_linear%s_workspace_bytes" % sfx, h_ptr, n_g, k, width, impl, ctypes.byref(ws_bytes))
        ws = torch.empty(max(ws_bytes.value, 1), dtype=torch.uint8, device=out.device)
        _lib.call("hgt_typed_linear" + sfx, a.data_ptr(), lda, w.data_ptr(), _lib.ptr(bias), k, width, g_ptr, h_ptr,
                  n_g, c_dev.data_ptr(), out.data_ptr(), impl, ws.data_ptr(), ws.numel(), st)

    @staticmethod
    def _presplit_linear(a_hi, a_lo, w, bias, k, width, table, out, st, groups=None):
        """hgt_typed_linear_presplit (bf16 `out`: hgt_typed_linear_presplit_bf16) over the table's groups, or the range
        `groups` = (first, count) of them."""
        g_dev, g_host, n_g, c_dev = table
        first, n_g = (0, n_g) if groups is None else groups
        g_ptr, h_ptr = g_dev.data_ptr() + first * g_host.itemsize, g_host.ctypes.data + first * g_host.itemsize
        sfx = "_bf16" if out.dtype == torch.bfloat16 else ""
        wsb = ctypes.c_size_t()
        _lib.call("hgt_typed_linear_presplit%s_workspace_bytes" % sfx, h_ptr, n_g, k, width, ctypes.byref(wsb))
        ws = torch.empty(max(wsb.value, 1), dtype=torch.uint8, device=out.device)
        _lib.call("hgt_typed_linear_presplit" + sfx, a_hi.data_ptr(), a_lo.data_ptr(), w.data_ptr(), _lib.ptr(bias), k,
                  width, g_ptr, h_ptr, n_g, c_dev.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(), st)

    def _kv_bf16(self):
        """Whether this layer stores its K'/V' tables as bf16 (kv_dtype).  Raises ValueError for a dtype it does not
        offer, before anything is launched."""
        dt = self.kv_dtype
        if dt == torch.float32:
            return False
        if dt != torch.bfloat16:
            raise ValueError("%s.kv_dtype must be torch.float32 or torch.bfloat16, got %r" % (type(self).__name__, dt))
        if not type(self)._has_skip:
            raise ValueError("DenseHGTConv has no bf16 K'/V' mode: set kv_dtype = torch.float32")
        return True

    def _check_inputs(self, node_inp, edge_time):
        if node_inp.device.type != "cuda":
            raise _lib.HgtError("pyhgt_b200.HGTConv runs on CUDA tensors only (got %s): there is no CPU "
                                "fallback" % node_inp.device)
        if node_inp.dtype != torch.float32:
            raise ValueError("node_inp must be float32 (the reference is fp32 throughout), got %s" % node_inp.dtype)
        if node_inp.dim() != 2 or node_inp.shape[1] != self.in_dim:
            raise ValueError("node_inp must be [N, %d], got %s" % (self.in_dim, tuple(node_inp.shape)))
        if self.in_dim != self.out_dim:
            # conv.py:131 adds node_inp to the out_dim-wide transform: the reference itself needs in == out
            raise ValueError("HGTConv needs in_dim == out_dim for the skip connection (conv.py:131)")
        if self.use_RTE and edge_time is None:
            raise ValueError("use_RTE=True needs edge_time (conv.py:91-92)")
        if self.out_dim % self.n_heads != 0:
            raise ValueError("out_dim=%d is not divisible by n_heads=%d" % (self.out_dim, self.n_heads))

    def forward(self, node_inp, node_type, edge_index, edge_type, edge_time=None):
        self._check_inputs(node_inp, edge_time)
        kv_bf16 = self._kv_bf16()
        if torch.is_grad_enabled() and (node_inp.requires_grad or any(p.requires_grad for p in self.parameters())):
            if kv_bf16:
                raise ValueError("kv_dtype=torch.bfloat16 is an inference mode and has no backward: run the layer "
                                 "under torch.no_grad() / torch.inference_mode(), or set kv_dtype = torch.float32")
            from .autograd import hgt_conv_autograd
            return hgt_conv_autograd(self, node_inp, node_type, edge_index, edge_type, edge_time)
        out, att, _ = self._forward_impl(node_inp, node_type, edge_index, edge_type, edge_time,
                                         want_att=self.keep_att, save=False)
        self.att = att
        return out

    # ------------------------------------------------------------------------------------------
    def _forward_fused(self, node_inp, node_type, edge_index, edge_type, edge_time, want_att,
                       active_per_type=None, out_map=None, out_rows=None, x_split=None, kv_runs=None):
        """Inference through the single entry point hgt_conv_forward (csrc/layer.cu).  The argument block is cached per
        (plan tables, parameter locations); per call only the data pointers change."""
        dev = node_inp.device
        d_in, d, H, T, R = self.in_dim, self.out_dim, self.n_heads, self.num_types, self.num_relations
        plan = _plan.get_plan(node_type, edge_index, edge_type, edge_time if self.use_RTE else None, T, R)
        N, E = plan.n_nodes, plan.n_edges
        if node_inp.shape[0] != N:
            raise ValueError("node_inp has %d rows but node_type has %d" % (node_inp.shape[0], N))
        kv_bf16 = self._kv_bf16()
        lt = _plan.layer_tables(plan, d_in, d, active_per_type, kv_runs, kv_bf16)
        tabs = [self._ptrs("wq", [l.weight for l in self.q_linears], dev),
                self._ptrs("bq", [l.bias for l in self.q_linears], dev),
                self._ptrs("wk", [l.weight for l in self.k_linears], dev),
                self._ptrs("bk", [l.bias for l in self.k_linears], dev),
                self._ptrs("wv", [l.weight for l in self.v_linears], dev),
                self._ptrs("bv", [l.bias for l in self.v_linears], dev),
                self._ptrs("wa", [l.weight for l in self.a_linears], dev),
                self._ptrs("ba", [l.bias for l in self.a_linears], dev)]
        if self.use_norm:
            tabs += [self._ptrs("nw", [n.weight for n in self.norms], dev), self._ptrs("nb", [n.bias for n in self.norms], dev)]
        scalars = [self.relation_att, self.relation_msg, self.relation_pri, self.skip]
        if self.use_RTE:
            scalars += [self.emb.emb.weight, self.emb.lin.weight, self.emb.lin.bias]
        key = (id(lt), kv_bf16) + tuple(t.data_ptr() for t in tabs) + tuple(t.data_ptr() for t in scalars)
        cache = self.__dict__.setdefault("_args_cache", {})
        ent = cache.get(key)
        if ent is None:
            a = _lib.ConvArgs()
            a.n_nodes, a.n_edges, a.kv_rows, a.cat_rows = N, E, plan.kv_rows, lt.cat_rows
            a.q_off, a.kv_off, a.proj_elems = lt.q_off, lt.kv_off, lt.proj_elems
            a.num_types, a.num_relations, a.n_heads, a.d_in, a.d_out, a.n_pairs = T, R, H, d_in, d, plan.n_pairs
            a.use_rte, a.use_norm = int(self.use_RTE), int(self.use_norm)
            a.kv_bf16, a.n_q_groups = int(kv_bf16), lt.n_q_groups
            a.n_tiles, a.n_split, a.n_hubs = plan.n_tiles, plan.n_split, plan.n_hubs
            a.perm = None if plan.sorted_types else plan.perm.data_ptr()
            a.type_row0 = plan.type_row0_dev.data_ptr()
            a.type_active = _lib.ptr(lt.type_active_dev)
            a.row_ptr, a.kv_row = plan.row_ptr.data_ptr(), plan.kv_row.data_ptr()
            a.rte_row = plan.rte_row.data_ptr() if self.use_RTE else None
            a.csr_eid, a.tiles, a.hubs = plan.csr_eid.data_ptr(), plan.tiles.data_ptr(), plan.hubs.data_ptr()
            a.d_tile_counts = _lib.ptr(plan.tile_counts_dev)
            a.pair_type, a.pair_rel = plan.pair_type_dev.data_ptr(), plan.pair_rel_dev.data_ptr()
            a.cat_row0, a.q_row0 = lt.cat_row0_dev.data_ptr(), lt.q_row0_dev.data_ptr()
            for name, tab in (("proj", lt.proj_groups), ("rte", lt.rte_groups), ("rt", lt.rt_group), ("upd", lt.upd_groups)):
                g_dev, g_host, n_g, c_dev = tab
                setattr(a, name + "_groups", g_dev.data_ptr())
                setattr(a, "h_" + name + "_groups", g_host.ctypes.data)
                setattr(a, name + "_cblocks", c_dev.data_ptr())
                if name != "rt":
                    setattr(a, "n_" + name + "_groups", n_g)
            (a.wq, a.bq, a.wk, a.bk, a.wv, a.bv, a.wa, a.ba) = [t.data_ptr() for t in tabs[:8]]
            if self.use_norm:
                a.norm_w, a.norm_b = tabs[8].data_ptr(), tabs[9].data_ptr()
            a.relation_att, a.relation_msg = self.relation_att.data_ptr(), self.relation_msg.data_ptr()
            a.relation_pri, a.skip = self.relation_pri.data_ptr(), self.skip.data_ptr()
            if self.use_RTE:
                a.emb_weight, a.emb_lin_w = self.emb.emb.weight.data_ptr(), self.emb.lin.weight.data_ptr()
                a.emb_lin_b = self.emb.lin.bias.data_ptr()
            if len(cache) >= 4:                                    # entries pin their plan: keep only a few
                cache.clear()
            ent = cache[key] = (a, lt, plan, tabs)                 # keep the tables the pointers refer to alive
        a = ent[0]
        x = node_inp.contiguous()
        if x_split is None and plan.sorted_types and self.linear_impl in (0, 2):
            hint = getattr(node_inp, "_hgt_split", None)
            if (hint is not None and hint[2] == node_inp._version and x is node_inp
                    and tuple(hint[0].shape) == (N, d_in) and d_in % 16 == 0 and d_in >= 64):
                x_split = (hint[0], hint[1])
        a.edge_variant, a.linear_impl = self.edge_variant, self.linear_impl
        a.x = x.data_ptr()
        a.x_hi, a.x_lo = (x_split[0].data_ptr(), x_split[1].data_ptr()) if x_split is not None else (None, None)
        if out_map is not None and not plan.sorted_types:
            raise ValueError("out_map needs a type-sorted node order")
        a.out_map = _lib.ptr(out_map)
        out = torch.empty((N if out_rows is None else out_rows, d), dtype=torch.float32, device=dev)
        att = torch.empty((E, H), dtype=torch.float32, device=dev) if want_att else None
        a.out, a.att = out.data_ptr(), _lib.ptr(att)
        o_hi = o_lo = None
        if (self.emit_split and plan.sorted_types and out_map is None and lt.type_active_dev is None and d % 16 == 0
                and d >= 64):
            o_hi = torch.empty((N, d), dtype=torch.bfloat16, device=dev)
            o_lo = torch.empty((N, d), dtype=torch.bfloat16, device=dev)
        a.out_hi, a.out_lo = _lib.ptr(o_hi), _lib.ptr(o_lo)
        wsb = ctypes.c_size_t()
        _lib.call("hgt_conv_workspace_bytes", ctypes.byref(a), ctypes.byref(wsb))
        ws = torch.empty(wsb.value, dtype=torch.uint8, device=dev)
        _lib.call("hgt_conv_forward", ctypes.byref(a), ws.data_ptr(), ws.numel(), _stream())
        if o_hi is not None:
            out._hgt_split = (o_hi, o_lo, out._version)
        return out, att, None

    def _forward_impl(self, node_inp, node_type, edge_index, edge_type, edge_time, want_att, save,
                      active_per_type=None, out_map=None, out_rows=None, x_split=None, kv_runs=None):
        """out_map / out_rows (sharded runs): int32 [N] map from rank-order row to output row and the number of output
        rows; rows that are not active (halo sources) are never written, so the output holds exactly the owned rows."""
        if save and self._kv_bf16():
            raise ValueError("kv_dtype=torch.bfloat16 is an inference mode: nothing is saved for a backward pass")
        if (self.fused_call and not save and HGTConv.event_sink is None and type(self)._has_skip
                and not (self.training and self.drop.p > 0)):
            return self._forward_fused(node_inp, node_type, edge_index, edge_type, edge_time, want_att,
                                       active_per_type, out_map, out_rows, x_split, kv_runs)
        c = self._core(node_inp, node_type, edge_index, edge_type, edge_time, want_att, save, active_per_type,
                       gelu_before_a=True, x_split=x_split, kv_runs=kv_runs)
        plan, lt, o, x_sorted, N, d, T, st = c["plan"], c["lt"], c["o"], c["x_sorted"], c["N"], c["d"], c["T"], c["st"]
        f32 = dict(dtype=torch.float32, device=o.device)
        norm_w = norm_b = None
        if self.use_norm:
            norm_w = torch.stack([n.weight for n in self.norms]).contiguous()
            norm_b = torch.stack([n.bias for n in self.norms]).contiguous()
        out = torch.empty((N if out_rows is None else out_rows, d), **f32)
        if out_map is not None:
            if not plan.sorted_types:
                raise ValueError("out_map needs a type-sorted node order")
            perm_ptr = out_map.data_ptr()
        else:
            perm_ptr = None if plan.sorted_types else plan.perm.data_ptr()
        o_hi = o_lo = None
        if (self.emit_split and perm_ptr is None and lt.type_active_dev is None and d % 16 == 0 and d >= 64
                and not self.training):
            o_hi = torch.empty((N, d), dtype=torch.bfloat16, device=o.device)
            o_lo = torch.empty((N, d), dtype=torch.bfloat16, device=o.device)
        with self._stage("update_epilogue"):
            _lib.call("hgt_update_epilogue", o.data_ptr(), x_sorted.data_ptr(), plan.type_row0_dev.data_ptr(), T,
                      self.skip.data_ptr(), _lib.ptr(norm_w), _lib.ptr(norm_b), perm_ptr,
                      _lib.ptr(lt.type_active_dev), N, d, out.data_ptr(), _lib.ptr(o_hi), _lib.ptr(o_lo), st)
        if o_hi is not None:
            out._hgt_split = (o_hi, o_lo, out._version)          # consumed by the next layer's projection (see _core)
        return out, c["att"], (c if save else None)

    def _core(self, node_inp, node_type, edge_index, edge_type, edge_time, want_att, save, active_per_type,
              gelu_before_a, x_split=None, kv_runs=None):
        """Everything up to and including the typed a_linear: plan, weight fold, typed projections, fused edge kernel
        (gelu fused iff gelu_before_a and not save), a_linears.  Returns a dict of the intermediates."""
        dev = node_inp.device
        d_in, d = self.in_dim, self.out_dim
        H, T, R = self.n_heads, self.num_types, self.num_relations
        st = _stream()
        plan = _plan.get_plan(node_type, edge_index, edge_type, edge_time if self.use_RTE else None, T, R)
        N, E, P = plan.n_nodes, plan.n_edges, plan.n_pairs
        if node_inp.shape[0] != N:
            raise ValueError("node_inp has %d rows but node_type has %d" % (node_inp.shape[0], N))
        kv_bf16 = self._kv_bf16()
        lt = _plan.layer_tables(plan, d_in, d, active_per_type, kv_runs, kv_bf16)
        f32 = dict(dtype=torch.float32, device=dev)
        x = node_inp.contiguous()
        if x_split is None and plan.sorted_types and self.linear_impl in (0, 2):
            hint = getattr(node_inp, "_hgt_split", None)            # left by the previous layer's update epilogue
            if (hint is not None and hint[2] == node_inp._version and x is node_inp
                    and tuple(hint[0].shape) == (N, d_in) and d_in % 16 == 0 and d_in >= 64):
                x_split = (hint[0], hint[1])
        if plan.sorted_types:
            x_sorted = x
        else:
            with self._stage("gather_rows"):
                x_sorted = torch.empty_like(x)
                _lib.call("hgt_gather_rows", x.data_ptr(), plan.perm.data_ptr(), N, d_in, x_sorted.data_ptr(), st)

        # 1. fold relation matrices into the typed K/V weights
        w_cat = torch.empty((max(lt.cat_rows, 1), d_in), **f32)
        b_cat = torch.empty(max(lt.cat_rows, 1), **f32)
        wq = self._ptrs("wq", [l.weight for l in self.q_linears], dev)
        bq = self._ptrs("bq", [l.bias for l in self.q_linears], dev)
        wk = self._ptrs("wk", [l.weight for l in self.k_linears], dev)
        bk = self._ptrs("bk", [l.bias for l in self.k_linears], dev)
        wv = self._ptrs("wv", [l.weight for l in self.v_linears], dev)
        bv = self._ptrs("bv", [l.bias for l in self.v_linears], dev)
        _lib.call("hgt_fold_weights", wq.data_ptr(), bq.data_ptr(), wk.data_ptr(), bk.data_ptr(), wv.data_ptr(),
                  bv.data_ptr(), self.relation_att.data_ptr(), self.relation_msg.data_ptr(),
                  self.relation_pri.data_ptr(), T, R, H, d_in, d, P, plan.pair_type_dev.data_ptr(),
                  plan.pair_rel_dev.data_ptr(), lt.cat_row0_dev.data_ptr(), lt.q_row0_dev.data_ptr(),
                  w_cat.data_ptr(), b_cat.data_ptr(), st)

        # 2. typed projections: Q [N,d] and the folded [K'|V'] table (+ trailing all-zero row); with bf16 tables the Q
        #    groups and the K'/V' groups are two calls into two buffers
        kv_f = dict(dtype=torch.bfloat16, device=dev) if kv_bf16 else f32
        proj = torch.empty(lt.proj_elems, **f32)
        q_tab = proj[lt.q_off:lt.q_off + N * d]
        kv_tab = torch.empty(lt.kv_elems, **kv_f) if kv_bf16 else proj[lt.kv_off:]
        kv_tab[plan.kv_rows * 2 * d:].zero_()
        n_g = lt.proj_groups[2]
        parts = [((0, lt.n_q_groups), proj), ((lt.n_q_groups, n_g - lt.n_q_groups), kv_tab)] if kv_bf16 else [(None, proj)]
        pre = x_split if plan.sorted_types else None
        with self._stage("proj_linear"):
            if kv_bf16 and pre is None and self.linear_impl in (0, 2) and d_in % 16 == 0 and d_in >= 64:
                # two tensor-core GEMMs over the same x: split it once (the GEMM's own split, so the same bits)
                pre = (torch.empty((N, d_in), dtype=torch.bfloat16, device=dev),
                       torch.empty((N, d_in), dtype=torch.bfloat16, device=dev))
                _lib.call("hgt_act_split", x_sorted.data_ptr(), d_in, N, d_in, 0, None, pre[0].data_ptr(),
                          pre[1].data_ptr(), st)
            for groups, dst in parts:
                if pre is not None:
                    # A operand already split by its producer (the fused halo pull): tensor-core GEMM without the split
                    # pass
                    self._presplit_linear(pre[0], pre[1], w_cat, b_cat, d_in, d, lt.proj_groups, dst, st, groups)
                else:
                    self._typed_linear(x_sorted, d_in, w_cat, b_cat, d_in, d, lt.proj_groups, dst, self.linear_impl, st,
                                       groups)
        kvr = None
        if self.use_RTE:
            # RT = lin(emb.weight) [240,d] (conv.py:299), then projected with every pair's K'/V' weights (no bias)
            rt = torch.empty((_plan.RTE_MAX_LEN, d_in), **f32)
            self._typed_linear(self.emb.emb.weight, d_in, self.emb.lin.weight, self.emb.lin.bias, d_in, d_in,
                               lt.rt_group, rt, 1, st)
            kvr = torch.empty((P * _plan.RTE_MAX_LEN + 1) * 2 * d, **kv_f)
            kvr[P * _plan.RTE_MAX_LEN * 2 * d:].zero_()
            self._typed_linear(rt, d_in, w_cat, None, d_in, d, lt.rte_groups, kvr, 1, st)

        # 3. fused edge kernel -> gelu(aggregate)
        ws_bytes = ctypes.c_size_t()
        _lib.call("hgt_edge_workspace_bytes", plan.n_split, d, H, ctypes.byref(ws_bytes))
        ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=dev)
        # When the a_linear GEMM will run on the tensor cores, the edge kernel writes gelu(agg) directly as the bf16
        # hi/lo operand split (no fp32 round trip, no separate split pass).
        fuse_split = (gelu_before_a and not save and self.linear_impl in (0, 2) and d % 16 == 0 and d >= 64
                      and not (self.training and self.drop.p > 0))
        g_act = None if fuse_split else torch.empty((N, d), **f32)
        g_hi = torch.empty((N, d), dtype=torch.bfloat16, device=dev) if fuse_split else None
        g_lo = torch.empty((N, d), dtype=torch.bfloat16, device=dev) if fuse_split else None
        att = torch.empty((E, H), **f32) if want_att else None
        stats = torch.empty((N, 2 * H), **f32) if save else None
        with self._stage("edge"):
            _lib.call("hgt_edge_forward_bf16kv" if kv_bf16 else "hgt_edge_forward", q_tab.data_ptr(), kv_tab.data_ptr(), _lib.ptr(kvr), plan.row_ptr.data_ptr(),
                      plan.kv_row.data_ptr(), _lib.ptr(plan.rte_row) if self.use_RTE else None,
                      plan.csr_eid.data_ptr(), plan.tiles.data_ptr(), plan.n_tiles, plan.n_split,
                      plan.hubs.data_ptr(), plan.n_hubs, N, E, d, H, 1 if (gelu_before_a and not save) else 0,
                      _lib.ptr(g_act), _lib.ptr(att), _lib.ptr(stats), _lib.ptr(g_hi), _lib.ptr(g_lo), ws.data_ptr(),
                      ws.numel(), self.edge_variant, _lib.ptr(plan.tile_counts_dev), plan.type_row0_dev.data_ptr(), T,
                      _lib.ptr(lt.type_active_dev), st)

        # 4. typed output linear (conv.py:125 / conv.py:261)
        agg = None
        if save or not gelu_before_a:
            agg = g_act
            g_act = F.gelu(agg) if gelu_before_a else agg
        wa_cat = torch.empty((T * d, d), **f32)
        ba_cat = torch.empty(T * d, **f32)
        wa = self._ptrs("wa", [l.weight for l in self.a_linears], dev)
        ba = self._ptrs("ba", [l.bias for l in self.a_linears], dev)
        _lib.call("hgt_concat_linears", wa.data_ptr(), ba.data_ptr(), T, d, d, wa_cat.data_ptr(), ba_cat.data_ptr(), st)
        o = torch.empty((N, d), **f32)
        with self._stage("upd_linear"):
            if fuse_split:
                self._presplit_linear(g_hi, g_lo, wa_cat, ba_cat, d, d, lt.upd_groups, o, st)
            else:
                self._typed_linear(g_act, d, wa_cat, ba_cat, d, d, lt.upd_groups, o, self.linear_impl, st)
        if self.training and self.drop.p > 0:
            o = self.drop(o)                                       # conv.py:125 (train mode only)
        return dict(plan=plan, lt=lt, x_sorted=x_sorted, w_cat=w_cat, proj=proj, kvr=kvr, agg=agg, o=o, stats=stats,
                    att=att, N=N, d=d, T=T, st=st)


class DenseHGTConv(HGTConv):
    """Reference conv.py:143-280: the same message() as HGTConv (same typed projections, relation transforms,
    softmax by destination, aggregation => the same CUDA kernels), but update() is
        y = LayerNorm_t(a_linear_t(agg) + x)                         (no gelu, no skip gate; conv.py:261-266)
        out = out_norm(out_linear(gelu(mid_linear(y))) + y)          (shared 2-layer FFN; conv.py:273-274)
    Every stage runs through the C ABI (autograd.dense_hgt_forward): typed tcgen05 GEMMs with the FFN's gelu inside the
    operand split, the residual + LayerNorm in `hgt_update_epilogue`'s residual mode; training uses the same native backward
    kernels as HGTConv.  Parameter names match the reference (mid_linear, out_linear, out_norm; no `skip`)."""
    _has_skip = False

    def __init__(self, in_dim, out_dim, num_types, num_relations, n_heads, dropout=0.2, use_norm=True,
                 use_RTE=True, **kwargs):
        super().__init__(in_dim, out_dim, num_types, num_relations, n_heads, dropout, use_norm, use_RTE, **kwargs)
        self.mid_linear = nn.Linear(out_dim, out_dim * 2)
        self.out_linear = nn.Linear(out_dim * 2, out_dim)
        self.out_norm = nn.LayerNorm(out_dim)

    def forward(self, node_inp, node_type, edge_index, edge_type, edge_time=None):
        self._check_inputs(node_inp, edge_time)
        self._kv_bf16()                                            # raises for bf16: this layer has no such mode
        from .autograd import dense_hgt_forward
        return dense_hgt_forward(self, node_inp, node_type, edge_index, edge_type, edge_time)


class GeneralConv(nn.Module):
    """String-keyed dispatch, reference conv.py:303-323.  'hgt' and 'dense_hgt' resolve to the CUDA layers above;
    'gcn' / 'gat' are PyG library layers, not this path (SURVEY.md §8f), and raise."""

    def __init__(self, conv_name, in_hid, out_hid, num_types, num_relations, n_heads, dropout, use_norm=True,
                 use_RTE=True):
        super().__init__()
        self.conv_name = conv_name
        if self.conv_name == 'hgt':
            self.base_conv = HGTConv(in_hid, out_hid, num_types, num_relations, n_heads, dropout, use_norm, use_RTE)
        elif self.conv_name == 'dense_hgt':
            self.base_conv = DenseHGTConv(in_hid, out_hid, num_types, num_relations, n_heads, dropout, use_norm,
                                          use_RTE)
        else:
            raise NotImplementedError("pyhgt_b200 implements conv_name 'hgt' and 'dense_hgt' only (got %r)" % conv_name)

    def forward(self, meta_xs, node_type, edge_index, edge_type, edge_time):
        return self.base_conv(meta_xs, node_type, edge_index, edge_type, edge_time)


def set_kv_dtype(module, dtype):
    """Set `kv_dtype` on every HGTConv in `module`'s tree (e.g. a GNN) and return `module`.

    torch.bfloat16 stores the folded K'/V' tables in bf16 for inference (about half the edge kernel's memory traffic and
    half the table memory); torch.float32 is the default, exact fp32 path.  The attribute is a plain instance attribute:
    state_dict and pickling are unchanged."""
    if dtype not in (torch.float32, torch.bfloat16):
        raise ValueError("kv_dtype must be torch.float32 or torch.bfloat16, got %r" % (dtype,))
    for m in module.modules():
        if isinstance(m, HGTConv):
            m.kv_dtype = dtype
    return module
