"""Per-graph plan for the HGTConv hot path: what PyG's ``propagate`` and the reference's T*T*R boolean
triple masks (pyHGT/conv.py:57,71-84) recompute every layer is built ONCE per graph here, on the GPU,
through the C ABI (hgt_plan_*):

  * type-sorted node order (rank / perm, per-type row ranges),
  * destination-sorted CSR (row_ptr, csr_eid) of the int64 COO ``edge_index`` (row 0 = source,
    row 1 = target: pyHGT/data.py:245,254),
  * the <source_type, relation> "pairs" that occur, and for every CSR edge the row of its source in the
    folded [K'|V'] table (kv_row) and in the RTE table (rte_row),
  * cost-balanced work tiles (hub destinations split) for the fused edge kernel.

Plans are cached per (node_type, edge_index, edge_type, edge_time) tensor identity, so the layers of a
GNN stack (pyHGT/model.py:78-79 passes the same tensors to every layer) share one plan.
"""
import ctypes
import os
import weakref
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib

RTE_MAX_LEN = 240            # conv.py:287
TILE_TARGET_EDGES = int(os.environ.get("HGT_TILE_EDGES", "64"))       # edges per work tile (cost units: csrc/plan.cu)
TILE_SPLIT_EDGES = int(os.environ.get("HGT_SPLIT_EDGES", "1024"))     # larger destinations are split across warps


def _stream():
    return torch.cuda.current_stream().cuda_stream


@dataclass
class GraphPlan:
    n_nodes: int
    n_edges: int
    num_types: int
    num_relations: int
    has_time: bool
    sorted_types: bool
    rank: torch.Tensor            # [N] int32
    perm: torch.Tensor            # [N] int32
    type_count: list              # [T+1] host ints (bucket T = out-of-range types)
    type_row0: list               # [T+2] host prefix
    type_row0_dev: torch.Tensor   # [T+2] int32
    row_ptr: torch.Tensor         # [N+1] int32
    csr_eid: torch.Tensor         # [E] int32
    kv_row: torch.Tensor          # [E] int32
    rte_row: torch.Tensor         # [E] int32 or None
    pairs: list                   # [(src_type, relation)]
    pair_row0: list               # first KV row of each pair
    kv_rows: int                  # rows in the KV table, excluding the trailing zero row
    tiles: torch.Tensor           # [n_tiles,4] int32
    n_tiles: int
    n_split: int
    hubs: torch.Tensor = None     # [n_hubs,4] int32 {dst, first partial slot, pieces, 0}
    n_hubs: int = 0
    pair_type_dev: torch.Tensor = None
    pair_rel_dev: torch.Tensor = None
    tile_counts_dev: torch.Tensor = None   # sync-free plans: device {n_tiles, n_split, n_hubs}; the host fields are bounds
    flags_dev: torch.Tensor = None         # sync-free plans: range-check flags left on the device (see check())
    _layer_tables: dict = field(default_factory=dict)
    _det: dict = field(default_factory=dict)  # deterministic backward: source-major indices (det_index)

    def check(self):
        """Sync-free plans defer the index range checks: this reads the flags back (one host sync) and raises like
        the synchronous build does."""
        if self.flags_dev is not None:
            f = self.flags_dev.cpu()
            if int(f[0]) != 0:
                raise IndexError("edge_index contains node ids outside [0, %d)" % self.n_nodes)
            if self.has_time and int(f[1]) != 0:
                raise IndexError("edge_time contains values outside [0, %d) (RelTemporalEncoding table size)" % RTE_MAX_LEN)

    @property
    def n_pairs(self):
        return len(self.pairs)


_CACHE = []          # [(weakrefs, versions, key_extra, plan)], most recent last
_CACHE_SIZE = 8


def _cache_lookup(tensors, extra):
    for entry in reversed(_CACHE):
        refs, versions, ex, plan = entry
        if ex != extra:
            continue
        ok = True
        for i, (r, v, t) in enumerate(zip(refs, versions, tensors)):
            if i == 3 and t is None and r is not None and r() is not None:
                continue          # a plan built WITH edge_time also serves a layer that does not use it (use_RTE=False)
            if (r is None) != (t is None):
                ok = False
                break
            if r is not None and (r() is not t or t._version != v):
                ok = False
                break
        if ok:
            return plan
    return None


def _cache_store(tensors, extra, plan):
    refs = [None if t is None else weakref.ref(t) for t in tensors]
    versions = [None if t is None else t._version for t in tensors]
    _CACHE.append((refs, versions, extra, plan))
    if len(_CACHE) > _CACHE_SIZE:
        _CACHE.pop(0)


def clear_plan_cache():
    _CACHE.clear()


def _as_i64(t, name, device):
    if t is None:
        return None
    if t.device != device:
        raise ValueError("%s is on %s but node features are on %s" % (name, t.device, device))
    if t.dtype != torch.int64:
        # the reference feeds LongTensors everywhere (data.py:252-255); no silent truncation
        raise ValueError("%s must be int64 (torch.LongTensor), got %s" % (name, t.dtype))
    return t.contiguous()


_PIN_KEEP = None     # a list while a CUDA graph is being captured (graphed.py): captured H2D copies re-read their pinned
                     # sources at every replay, so those must outlive the capture


def _to_dev_async(arr, dev):
    """Small host table -> device through pinned staging, without synchronising the stream."""
    t = torch.from_numpy(arr)
    if dev.type == "cuda":
        pinned = t.pin_memory()
        if _PIN_KEEP is not None:
            _PIN_KEEP.append(pinned)
        return pinned.to(dev, non_blocking=True)
    return t.to(dev)


def rebuild_plan(node_type, edge_index, edge_type, edge_time, num_types, num_relations, host_meta):
    """Build the plan of these tensors NOW (dropping a cached one) and cache it: the layers called next find it.  Used by
    graphed.py so that the plan build itself lands inside the captured CUDA graph."""
    tensors = (node_type, edge_index, edge_type, edge_time)
    for i in range(len(_CACHE) - 1, -1, -1):
        refs = _CACHE[i][0]
        if all((r is None and t is None) or (r is not None and r() is t) for r, t in zip(refs, tensors)):
            _CACHE.pop(i)
    plan = build_plan(node_type, edge_index, edge_type, edge_time, num_types, num_relations, host_meta)
    _cache_store(tensors, (num_types, num_relations), plan)
    return plan


def get_plan(node_type, edge_index, edge_type, edge_time, num_types, num_relations, use_cache=True, host_meta=None):
    """`host_meta` (optional): what the host already knows about the graph — {"type_count": [T+1 ints], "sorted": bool,
    "pairs": [(source_type, relation), ...]} — e.g. from `data.to_torch`, which builds the tensors from per-type blocks.
    With it the plan is built WITHOUT any host read-back or stream synchronisation (sampled-subgraph regime: a new
    graph every batch, OAG/train_paper_field.py:241); index range checks are then deferred (GraphPlan.check())."""
    tensors = (node_type, edge_index, edge_type, edge_time)
    extra = (num_types, num_relations)
    if use_cache:
        hit = _cache_lookup(tensors, extra)
        if hit is not None:
            return hit
    plan = build_plan(node_type, edge_index, edge_type, edge_time, num_types, num_relations, host_meta)
    if use_cache:
        _cache_store(tensors, extra, plan)
    return plan


def build_plan(node_type, edge_index, edge_type, edge_time, num_types, num_relations, host_meta=None):
    dev = node_type.device
    if dev.type != "cuda":
        raise _lib.HgtError("pyhgt_b200 runs on CUDA tensors only (got %s); there is no CPU fallback" % dev)
    nt = _as_i64(node_type, "node_type", dev)
    ei = _as_i64(edge_index, "edge_index", dev)
    et = _as_i64(edge_type, "edge_type", dev)
    tm = _as_i64(edge_time, "edge_time", dev)
    N = nt.numel()
    if ei.dim() != 2 or ei.shape[0] != 2:
        raise ValueError("edge_index must have shape [2, E], got %s" % (tuple(ei.shape),))
    E = ei.shape[1]
    if et.numel() != E or (tm is not None and tm.numel() != E):
        raise ValueError("edge_type / edge_time must have one entry per edge (E=%d)" % E)
    if N >= 2 ** 31 - 1024 or E >= 2 ** 31 - 1024:
        raise ValueError("graph too large for int32 CSR indices (N=%d, E=%d)" % (N, E))
    T, R = int(num_types), int(num_relations)
    st = _stream()
    i32 = dict(dtype=torch.int32, device=dev)

    ws_bytes = ctypes.c_size_t()
    _lib.call("hgt_plan_workspace_bytes", N, E, ctypes.byref(ws_bytes))
    ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=dev)

    # one small buffer for everything the host may read back: [type_count T+1 | sorted 1 | presence T*R | flags 4]
    meta = torch.zeros(T + 1 + 1 + T * R + 4, **i32)
    type_count_d = meta[:T + 1]
    sorted_d = meta[T + 1:T + 2]
    presence_d = meta[T + 2:T + 2 + T * R]
    flags_d = meta[T + 2 + T * R:]
    sync_free = host_meta is not None
    if sync_free and host_meta.get("sorted", False):
        rank = torch.arange(max(N, 1), **i32)                  # type-contiguous layout (to_torch): identity order
        perm = rank
    else:
        rank = torch.empty(max(N, 1), **i32)
        perm = torch.empty(max(N, 1), **i32)
        _lib.call("hgt_plan_nodes", nt.data_ptr(), N, T, rank.data_ptr(), perm.data_ptr(), type_count_d.data_ptr(),
                  sorted_d.data_ptr(), ws.data_ptr(), ws.numel(), st)
    row_ptr = torch.empty(N + 1, **i32)
    csr_eid = torch.empty(max(E, 1), **i32)
    _lib.call("hgt_plan_edges_sort", ei.data_ptr(), et.data_ptr(), nt.data_ptr(), rank.data_ptr(), N, E, T, R,
              row_ptr.data_ptr(), csr_eid.data_ptr(), presence_d.data_ptr(), flags_d.data_ptr(), ws.data_ptr(),
              ws.numel(), st)
    if sync_free:
        type_count = [int(v) for v in host_meta["type_count"]]
        if len(type_count) == T:
            type_count.append(0)
        if len(type_count) != T + 1 or sum(type_count) != N:
            raise ValueError("host_meta['type_count'] must hold T (+1) counts summing to N=%d, got %s" % (N, type_count))
        sorted_types = bool(host_meta.get("sorted", False))
        presence = np.zeros((T, R), dtype=np.int32)
        for (s_, r_) in host_meta["pairs"]:
            if 0 <= s_ < T and 0 <= r_ < R:
                presence[s_, r_] = 1
    else:
        meta_h = meta.cpu().numpy()                       # the one host sync of the node/edge pass
        type_count = [int(v) for v in meta_h[:T + 1]]
        sorted_types = bool(meta_h[T + 1])
        presence = meta_h[T + 2:T + 2 + T * R].reshape(T, R)
        if meta_h[T + 2 + T * R] != 0:
            raise IndexError("edge_index contains node ids outside [0, %d)" % N)

    type_row0 = [0]
    for c in type_count:
        type_row0.append(type_row0[-1] + c)
    pairs, pair_row0, pair_of = [], [], -np.ones(T * R, dtype=np.int32)
    rows = 0
    for s in range(T):
        for r in range(R):
            if presence[s, r]:
                pair_of[s * R + r] = len(pairs)
                pairs.append((s, r))
                pair_row0.append(rows)
                rows += type_count[s]
    if rows >= 2 ** 31 - 1024:
        raise ValueError("folded K'/V' table needs %d rows: exceeds int32 row indices" % rows)
    P = len(pairs)
    small = np.concatenate([pair_of, np.asarray(pair_row0 + [0], dtype=np.int32)[:max(P, 1)],
                            np.asarray(type_row0, dtype=np.int32),
                            np.asarray([p[0] for p in pairs] + [0], dtype=np.int32)[:max(P, 1)],
                            np.asarray([p[1] for p in pairs] + [0], dtype=np.int32)[:max(P, 1)]]).astype(np.int32)
    small_d = _to_dev_async(small, dev)
    o = 0
    pair_of_d = small_d[o:o + T * R]; o += T * R
    pair_row0_d = small_d[o:o + max(P, 1)]; o += max(P, 1)
    type_row0_d = small_d[o:o + T + 2]; o += T + 2
    pair_type_d = small_d[o:o + max(P, 1)]; o += max(P, 1)
    pair_rel_d = small_d[o:o + max(P, 1)]

    kv_row = torch.empty(max(E, 1), **i32)
    rte_row = torch.empty(max(E, 1), **i32) if tm is not None else None
    _lib.call("hgt_plan_edges_fill", ei.data_ptr(), et.data_ptr(), _lib.ptr(tm), nt.data_ptr(), rank.data_ptr(),
              csr_eid.data_ptr(), N, E, T, R, pair_of_d.data_ptr(), pair_row0_d.data_ptr(), type_row0_d.data_ptr(),
              rows, P * RTE_MAX_LEN, kv_row.data_ptr(), _lib.ptr(rte_row), flags_d.data_ptr(), st)

    max_tiles = (2 * E + N) // (2 * TILE_TARGET_EDGES) + 3 * (E // TILE_SPLIT_EDGES) + 16
    tiles = torch.empty((max_tiles, 4), **i32)
    max_hubs = E // TILE_SPLIT_EDGES + 1
    hubs = torch.empty((max_hubs, 4), **i32)
    n_tiles_d = torch.zeros(4, **i32)
    if sync_free:
        # counts stay on the device; the host-side fields become the bounds the arrays were sized with
        _lib.call("hgt_plan_tiles", row_ptr.data_ptr(), N, E, TILE_TARGET_EDGES, TILE_SPLIT_EDGES, tiles.data_ptr(),
                  max_tiles, hubs.data_ptr(), max_hubs, n_tiles_d.data_ptr(), None, ws.data_ptr(), ws.numel(), st)
        has_hub = E > TILE_SPLIT_EDGES
        n_tiles = max_tiles if N > 0 else 0
        n_split = 2 * (E // TILE_SPLIT_EDGES) + 1 if has_hub else 0
        n_hubs = max_hubs if has_hub else 0
    else:
        n_tiles_h = (ctypes.c_int32 * 4)()
        _lib.call("hgt_plan_tiles", row_ptr.data_ptr(), N, E, TILE_TARGET_EDGES, TILE_SPLIT_EDGES, tiles.data_ptr(),
                  max_tiles, hubs.data_ptr(), max_hubs, n_tiles_d.data_ptr(), n_tiles_h, ws.data_ptr(), ws.numel(),
                  st)   # synchronises
        if tm is not None and int(flags_d[1].item()) != 0:
            raise IndexError("edge_time contains values outside [0, %d) (RelTemporalEncoding table size)" % RTE_MAX_LEN)
        n_tiles, n_split, n_hubs = int(n_tiles_h[0]), int(n_tiles_h[1]), int(n_tiles_h[2])
    return GraphPlan(n_nodes=N, n_edges=E, num_types=T, num_relations=R, has_time=tm is not None,
                     sorted_types=sorted_types, rank=rank, perm=perm, type_count=type_count, type_row0=type_row0,
                     type_row0_dev=type_row0_d, row_ptr=row_ptr, csr_eid=csr_eid, kv_row=kv_row, rte_row=rte_row,
                     pairs=pairs, pair_row0=pair_row0, kv_rows=rows, tiles=tiles[:max(n_tiles, 1)],
                     n_tiles=n_tiles, n_split=n_split, hubs=hubs[:max(n_hubs, 1)], n_hubs=n_hubs,
                     pair_type_dev=pair_type_d, pair_rel_dev=pair_rel_d,
                     tile_counts_dev=n_tiles_d if sync_free else None, flags_dev=flags_d if sync_free else None)


# ---- deterministic backward: source-major edge indices -------------------------------------------------------------

class TileIndex:
    """CSR positions grouped by a key (a [K'|V'] row or an RTE row), with work tiles over the groups.  Keeps the device
    arrays alive behind the `hgt_tile_set` handed to hgt_edge_backward_det."""

    def __init__(self, ptr, pos, tiles, hubs, counts, n_tiles, n_split, n_hubs):
        self.tensors = (ptr, pos, tiles, hubs, counts)
        self.c = _lib.TileSet(_lib.ptr(ptr), _lib.ptr(pos), tiles.data_ptr(), hubs.data_ptr(), _lib.ptr(counts),
                              n_tiles, n_split, n_hubs, 0)


def _group_index(key, E, n_keys, dev):
    """Group the E CSR positions by key[c] in [0, n_keys) (stable) and tile the groups like the destination CSR.  The
    tiler runs in its sync-free mode: counts stay on the device and the host fields are the bounds."""
    st = _stream()
    i32 = dict(dtype=torch.int32, device=dev)
    gb, pb = ctypes.c_size_t(), ctypes.c_size_t()
    _lib.call("hgt_plan_group_by_workspace_bytes", E, n_keys, ctypes.byref(gb))
    _lib.call("hgt_plan_workspace_bytes", n_keys, E, ctypes.byref(pb))
    ws = torch.empty(max(gb.value, pb.value), dtype=torch.uint8, device=dev)
    ptr = torch.empty(n_keys + 1, **i32)
    pos = torch.empty(max(E, 1), **i32)
    _lib.call("hgt_plan_group_by", key.data_ptr(), E, n_keys, ptr.data_ptr(), pos.data_ptr(), ws.data_ptr(), ws.numel(),
              st)
    max_tiles = (2 * E + n_keys) // (2 * TILE_TARGET_EDGES) + 3 * (E // TILE_SPLIT_EDGES) + 16
    max_hubs = E // TILE_SPLIT_EDGES + 1
    tiles = torch.empty((max_tiles, 4), **i32)
    hubs = torch.empty((max_hubs, 4), **i32)
    counts = torch.zeros(4, **i32)
    _lib.call("hgt_plan_tiles", ptr.data_ptr(), n_keys, E, TILE_TARGET_EDGES, TILE_SPLIT_EDGES, tiles.data_ptr(),
              max_tiles, hubs.data_ptr(), max_hubs, counts.data_ptr(), None, ws.data_ptr(), ws.numel(), st)
    has_hub = E > TILE_SPLIT_EDGES
    return TileIndex(ptr, pos, tiles, hubs, counts, max_tiles, 2 * (E // TILE_SPLIT_EDGES) + 1 if has_hub else 0,
                     max_hubs if has_hub else 0)


def det_index(plan, with_rte):
    """(csr_dst, destination index, [K'|V'] row index, RTE row index or None) for hgt_edge_backward_det, built on the
    first deterministic backward through this plan and cached on it.  Sync-free: nothing is read back to the host."""
    d = plan._det
    dev = plan.row_ptr.device
    E, N = plan.n_edges, plan.n_nodes
    if "src" not in d:
        d["csr_dst"] = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
        _lib.call("hgt_plan_csr_dst", plan.row_ptr.data_ptr(), N, E, d["csr_dst"].data_ptr(), _stream())
        d["dst"] = TileIndex(plan.row_ptr, None, plan.tiles, plan.hubs, plan.tile_counts_dev, plan.n_tiles, plan.n_split,
                             plan.n_hubs)
        d["src"] = _group_index(plan.kv_row, E, plan.kv_rows + 1, dev)
    if with_rte and "rte" not in d:
        d["rte"] = _group_index(plan.rte_row, E, plan.n_pairs * RTE_MAX_LEN + 1, dev)
    return d["csr_dst"], d["dst"], d["src"], d.get("rte") if with_rte else None


# ---- typed-linear descriptor tables (depend on the plan and on the layer's d_in / d_out) -------------

@dataclass
class LayerTables:
    cat_rows: int                 # rows of W_cat
    q_row0: list                  # [T] first W_cat row of W_q^t
    cat_row0: list                # [P] first W_cat row of pair p's K' block
    q_row0_dev: torch.Tensor
    cat_row0_dev: torch.Tensor
    proj_groups: tuple            # (groups_dev, groups_host_np, n_groups, cblocks_dev)
    rte_groups: tuple
    upd_groups: tuple
    rt_group: tuple               # RT = lin(emb.weight): one plain [240,d_in]x[d_in,d_in] group
    q_off: int                    # element offsets inside the projection buffer
    kv_off: int
    proj_elems: int
    type_active_dev: torch.Tensor = None


class GroupTable(tuple):
    """(groups_dev, groups_host, n_groups, cblocks_dev) plus `.c_host`, the host copy of the column-block table."""


def _pack_groups(groups, cblocks, dev):
    g = np.zeros(max(len(groups), 1), dtype=_lib.LIN_GROUP_DTYPE)
    for i, t in enumerate(groups):
        g[i] = t
    c = np.zeros(max(len(cblocks), 1), dtype=_lib.LIN_CBLOCK_DTYPE)
    for i, t in enumerate(cblocks):
        c[i] = t
    g_dev = _to_dev_async(g.view(np.uint8).copy(), dev)
    c_dev = _to_dev_async(c.view(np.uint8).copy(), dev)
    tab = GroupTable((g_dev, g, len(groups), c_dev))
    tab.c_host = c                 # host copy of the column-block table (the backward pass sizes its launches with it)
    return tab


def layer_tables(plan, d_in, d_out, active=None, kv_runs=None):
    """`active[t]` (sharded runs): only the first active[t] nodes of type t (in rank order) are destinations
    that need Q / a_linear / update; the rest of the type (halo sources) only get K'/V' rows.
    `kv_runs` (sharded runs): (((type, relation), ((row0, row1), ...)), ...) — type-relative row ranges whose K'/V' rows
    some local edge reads; the projection then covers those ranges only (the other rows of the table are never
    gathered and stay unwritten)."""
    key = (d_in, d_out, None if active is None else tuple(active), kv_runs)
    hit = plan._layer_tables.get(key)
    if hit is not None:
        return hit
    dev = plan.row_ptr.device
    T, P, N = plan.num_types, plan.n_pairs, plan.n_nodes
    pairs_of_type = [[] for _ in range(T)]
    for p, (s, _) in enumerate(plan.pairs):
        pairs_of_type[s].append(p)
    q_row0, cat_row0, rows = [], [0] * P, 0
    for t in range(T):
        q_row0.append(rows)
        for k, p in enumerate(pairs_of_type[t]):
            cat_row0[p] = rows + d_out + 2 * k * d_out
        rows += d_out * (1 + 2 * len(pairs_of_type[t]))
    q_off = 0
    kv_off = (N * d_out + 31) // 32 * 32                   # keep the KV table 128-byte aligned
    proj_elems = kv_off + (plan.kv_rows + 1) * 2 * d_out
    groups, cblocks = [], []
    act = [plan.type_count[t] if active is None else min(int(active[t]), plan.type_count[t]) for t in range(T)]
    for t in range(T):
        m = plan.type_count[t]
        if m == 0:
            continue
        a = act[t]
        if a > 0:
            first = len(cblocks)
            cblocks.append((q_off + plan.type_row0[t] * d_out, d_out))
            for p in pairs_of_type[t]:
                base = kv_off + plan.pair_row0[p] * 2 * d_out
                cblocks.append((base, 2 * d_out))
                cblocks.append((base + d_out, 2 * d_out))
            groups.append((plan.type_row0[t], a, q_row0[t], 1 + 2 * len(pairs_of_type[t]), first, 1))
        if m - a > 0 and pairs_of_type[t]:
            first = len(cblocks)
            for p in pairs_of_type[t]:
                base = kv_off + (plan.pair_row0[p] + a) * 2 * d_out
                cblocks.append((base, 2 * d_out))
                cblocks.append((base + d_out, 2 * d_out))
            groups.append((plan.type_row0[t] + a, m - a, q_row0[t] + d_out, 2 * len(pairs_of_type[t]), first, 1))
    if kv_runs is not None:
        # per-pair compaction: a Q group over the active prefix, and one K'/V' group per needed row range of every pair
        runs = dict(kv_runs)
        g2, c2 = [], []
        for t in range(T):
            if plan.type_count[t] and act[t] > 0:
                g2.append((plan.type_row0[t], act[t], q_row0[t], 1, len(c2), 1))
                c2.append((q_off + plan.type_row0[t] * d_out, d_out))
        for p, (s_, r_) in enumerate(plan.pairs):
            for (r0, r1) in runs.get((s_, r_), ()):
                r1 = min(int(r1), plan.type_count[s_])
                if r1 <= r0:
                    continue
                base = kv_off + (plan.pair_row0[p] + int(r0)) * 2 * d_out
                g2.append((plan.type_row0[s_] + int(r0), r1 - int(r0), cat_row0[p], 2, len(c2), 1))
                c2.append((base, 2 * d_out))
                c2.append((base + d_out, 2 * d_out))
        if len(g2) <= 64 and all((s_, r_) in runs for (s_, r_) in plan.pairs):
            groups, cblocks = g2, c2
    proj = _pack_groups(groups, cblocks, dev)
    # The backward's dX writes rows non-atomically, so it takes groups with DISJOINT row ranges: split the table into
    # such subsets (greedy interval colouring; the first subset writes dA, the others accumulate into it).
    subsets = []
    for gi, g_ in sorted(enumerate(groups), key=lambda t: (t[1][0], t[1][0] + t[1][1])):
        for sub in subsets:
            if all(g_[0] >= groups[o][0] + groups[o][1] or groups[o][0] >= g_[0] + g_[1] for o in sub):
                sub.append(gi)
                break
        else:
            subsets.append([gi])
    proj.bwd_tables = [proj] if len(subsets) <= 1 else [_pack_groups([groups[i] for i in sub], cblocks, dev)
                                                       for sub in subsets]
    groups, cblocks = [], []
    for p in range(P):
        first = len(cblocks)
        base = p * RTE_MAX_LEN * 2 * d_out
        cblocks.append((base, 2 * d_out))
        cblocks.append((base + d_out, 2 * d_out))
        groups.append((0, RTE_MAX_LEN, cat_row0[p], 2, first, 0))
    rte = _pack_groups(groups, cblocks, dev)
    groups, cblocks = [], []
    for t in range(T):
        m = act[t]
        if m == 0:
            continue
        groups.append((plan.type_row0[t], m, t * d_out, 1, len(cblocks), 1))
        cblocks.append((plan.type_row0[t] * d_out, d_out))
    upd = _pack_groups(groups, cblocks, dev)
    rt_group = _pack_groups([(0, RTE_MAX_LEN, 0, 1, 0, 1)], [(0, d_in)], dev)
    small = _to_dev_async(np.asarray(q_row0 + (cat_row0 if P else [0]) + act, dtype=np.int32), dev)
    lt = LayerTables(cat_rows=rows, q_row0=q_row0, cat_row0=cat_row0, q_row0_dev=small[:T],
                     cat_row0_dev=small[T:T + max(P, 1)],
                     type_active_dev=None if active is None else small[T + max(P, 1):], proj_groups=proj, rte_groups=rte, upd_groups=upd, rt_group=rt_group, q_off=q_off,
                     kv_off=kv_off, proj_elems=proj_elems)
    plan._layer_tables[key] = lt
    return lt
