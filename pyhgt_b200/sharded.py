"""Multi-GPU HGTConv: 1-D destination-node sharding with one all-to-all of halo source rows per layer
(SURVEY.md §8e; the reference itself is single-GPU — pyHGT has no distributed code).

Partition (built once per graph, identically on every rank from the full COO):
  * inside each node type the nodes are cut into `world` contiguous blocks balanced on the edge-kernel cost
    2*in_degree + 1, so every rank owns a slice of every type (typed GEMMs stay balanced) and ~E/world edges;
  * rank g keeps the in-edges of its owned destinations; the sources of those edges that it does not own
    are its halo.  Local node numbering = [owned (type-sorted) | halo (by owner, then global id)].
Per layer: gather the owned rows peers asked for -> ONE all_to_all_single (NCCL over NVLink on GPUs, gloo in
the CPU tests) straight into the tail of the local feature buffer -> the ordinary single-GPU kernels run on the
local graph, with Q / a_linear / update restricted to the owned rows and K'/V' projected for owned + halo.
"""
from dataclasses import dataclass

import torch
import torch.distributed as dist


def _require_fp32_kv(conv):
    """The sharded layer has fp32 K'/V' tables only (the bf16 mode of HGTConv.kv_dtype is single-GPU inference)."""
    if getattr(conv, "kv_dtype", torch.float32) != torch.float32:
        raise ValueError("the sharded path supports kv_dtype=torch.float32 only, got %r" % (conv.kv_dtype,))


def partition_owner(node_type, edge_index, num_types, world):
    """owner[n] in [0, world): contiguous cost-balanced blocks inside every node type (deterministic; runs on the device
    of its inputs)."""
    n = node_type.numel()
    wdev = node_type.device
    deg = torch.bincount(edge_index[1], minlength=n)
    cost = 2 * deg + 1
    owner = torch.zeros(n, dtype=torch.int64, device=wdev)
    for t in range(num_types):
        ids = (node_type == t).nonzero(as_tuple=True)[0]           # ascending ids = stable type order
        if ids.numel() == 0:
            continue
        c = cost[ids].cumsum(0)
        total = int(c[-1])
        # node i goes to block floor(prefix_before_i * world / total)
        before = c - cost[ids]
        owner[ids] = torch.clamp((before * world) // max(total, 1), max=world - 1)
    other = (node_type < 0) | (node_type >= num_types)
    if other.any():
        ids = other.nonzero(as_tuple=True)[0]
        owner[ids] = torch.arange(ids.numel(), device=wdev) * world // max(ids.numel(), 1)
    return owner


class _HaloExchange(torch.autograd.Function):
    """Differentiable halo exchange (NCCL / gloo path).  forward: owned rows -> local rows [per type: owned | halo].
    backward: the gradient of every halo row goes back to its owner with the REVERSE all-to-all and is added to the
    owner's row (a source feeds edges on several ranks), the gradient of owned rows stays local."""

    @staticmethod
    def forward(ctx, x_own, shard):
        ctx.shard = shard
        return shard._exchange_nccl(x_own)

    @staticmethod
    def backward(ctx, dx_local):
        sh = ctx.shard
        d = dx_local.shape[1]
        dx_local = dx_local.contiguous()
        d_cat = torch.empty_like(dx_local)
        d_cat.index_copy_(0, sh.cat_index.long(), dx_local)              # undo the [x_own | recv] -> local re-ordering
        d_own = d_cat[:sh.n_owned].clone()
        d_recv = d_cat[sh.n_owned:].contiguous()
        d_send = torch.empty((sh.send_idx.numel(), d), dtype=dx_local.dtype, device=dx_local.device)
        if sh.world > 1:
            dist.all_to_all_single(d_send, d_recv, sh.send_splits, sh.recv_splits, group=sh.group)
        d_own.index_add_(0, sh.send_idx, d_send)
        return d_own, None


@dataclass
class ShardedGraph:
    rank: int
    world: int
    device: torch.device
    n_owned: int
    n_halo: int
    n_local_edges: int
    owned_global: torch.Tensor        # [n_owned] global ids, type-sorted (CPU)
    halo_global: torch.Tensor         # [n_halo] global ids in all-to-all arrival order: by owner, then id (CPU)
    local_global: torch.Tensor        # [n_local] global id of every local row (CPU); local order = per type [owned | halo]
    node_type: torch.Tensor           # [n_local] local node types, non-decreasing (device)
    edge_index: torch.Tensor          # [2, E_local] local ids (device)
    edge_type: torch.Tensor
    edge_time: torch.Tensor
    send_idx: torch.Tensor            # [n_send] rows of x_own to send, grouped by destination rank
    send_splits: list
    recv_splits: list
    cat_index: torch.Tensor           # [n_local] int32: row of concat([x_own, recv]) for every local row
    pull_rank: torch.Tensor           # [n_local] int32: owner of every local row (P2P pull path)
    pull_row: torch.Tensor            # [n_local] int32: row inside the owner's x_own
    own_rows: torch.Tensor            # [n_owned] int64: local row of every owned node, in owned_global order
    active_per_type: list             # owned nodes of each type (type T = out-of-range bucket)
    max_owned: int                    # max n_owned over ranks (symmetric buffer rows)
    num_types: int
    num_relations: int
    group: object = None
    halo_mode: str = "auto"           # "nccl": one all_to_all_single per layer; "p2p": pull kernel over NVLink peer
                                      # memory; "auto": p2p on CUDA when symmetric memory works, else nccl
    pull_order: torch.Tensor = None   # [n_local] int32: processing order of the pull kernel (peers interleaved, staggered)
    _symm: object = None
    _slot: int = 0
    kv_runs: tuple = None             # (((type, relation), ((row0, row1), ...)), ...) type-relative local rows that need K'/V'

    @staticmethod
    def build(node_type, edge_index, edge_type, edge_time, num_types, num_relations, rank, world, device,
              group=None, halo_mode=None):
        import os
        # the O(N + E) passes below are plain tensor ops: run them on the target GPU when there is one (C2: 3.5 s on the
        # host cores vs a fraction of a second on the device); the id lists callers index host arrays with come back to
        # the CPU at the end
        wdev = torch.device(device) if torch.device(device).type == "cuda" else torch.device("cpu")
        node_type, edge_index, edge_type = node_type.to(wdev), edge_index.to(wdev), edge_type.to(wdev)
        edge_time = None if edge_time is None else edge_time.to(wdev)
        n = node_type.numel()
        i64 = dict(dtype=torch.int64, device=wdev)
        owner = partition_owner(node_type, edge_index, num_types, world)
        tkey = torch.where((node_type >= 0) & (node_type < num_types), node_type, torch.full_like(node_type, num_types))
        # position of every node inside its owner's (type-sorted) owned list — identical on every rank
        owned_pos = torch.empty(n, **i64)
        max_owned = 0
        owned = None
        for r in range(world):
            mine_r = (owner == r).nonzero(as_tuple=True)[0]
            owned_r = mine_r[torch.argsort(tkey[mine_r], stable=True)]
            owned_pos[owned_r] = torch.arange(owned_r.numel(), device=wdev)
            max_owned = max(max_owned, int(owned_r.numel()))
            if r == rank:
                owned = owned_r
        e_sel = (owner[edge_index[1]] == rank).nonzero(as_tuple=True)[0]    # in-edges of owned destinations
        src, dst = edge_index[0, e_sel], edge_index[1, e_sel]
        srcs = torch.unique(src)
        halo = srcs[owner[srcs] != rank]
        halo = halo[torch.argsort(owner[halo] * n + halo)]                   # arrival order: by owner, then id
        n_owned, n_halo = int(owned.numel()), int(halo.numel())
        # local order: per type [owned | halo]  => node_type is sorted, Q/update act on a prefix of every type.
        # Inside both parts the nodes are ordered by WHICH relations they feed on this rank (bit r of `rel_mask`: the
        # node is the source of a local edge of relation r), owned ascending / halo descending, so that the rows a
        # <source type, relation> pair really needs form a few contiguous runs: K'/V' are projected for those runs only
        # (kv_runs) instead of for every local node of the type.
        cat_ids = torch.cat([owned, halo])                                   # order of concat([x_own, recv])
        is_halo = torch.cat([torch.zeros(n_owned, **i64), torch.ones(n_halo, **i64)])
        rel_sel = edge_type[e_sel]
        rel_mask = torch.zeros(n, **i64)
        compact = num_relations <= 16
        if compact:
            for r in range(num_relations):
                sr = src[rel_sel == r]
                rel_mask[sr] = rel_mask[sr] | (1 << r)
        n_masks = 1 << min(num_relations, 16)
        mk = rel_mask[cat_ids]
        sub = torch.where(is_halo == 1, n_masks - 1 - mk, mk)
        order = torch.argsort((tkey[cat_ids] * 2 + is_halo) * n_masks + sub, stable=True)
        local_global = cat_ids[order]
        # runs of local rows (type-relative) whose mask contains relation r, per (type, relation)
        kv_runs = None
        if compact:
            kv_runs = {}
            lt_ = tkey[local_global]
            lm = rel_mask[local_global]
            for t in range(num_types):
                rows_t = (lt_ == t).nonzero(as_tuple=True)[0]
                if rows_t.numel() == 0:
                    continue
                mt = lm[rows_t]
                for r in range(num_relations):
                    has = ((mt >> r) & 1).to(torch.int8)
                    if int(has.sum()) == 0:
                        continue
                    z8 = torch.zeros(1, dtype=torch.int8, device=wdev)
                    edge_ = torch.diff(torch.cat([z8, has, z8]))
                    starts = (edge_ == 1).nonzero(as_tuple=True)[0].tolist()
                    ends = (edge_ == -1).nonzero(as_tuple=True)[0].tolist()
                    kv_runs[(t, r)] = tuple(zip(starts, ends))
        local_of = torch.full((n,), -1, **i64)
        local_of[local_global] = torch.arange(local_global.numel(), device=wdev)
        ei_local = torch.stack([local_of[src], local_of[dst]])
        recv_splits = torch.bincount(owner[halo], minlength=world).tolist()
        send_lists = []
        dst_owner_all = owner[edge_index[1]]
        src_owner_all = owner[edge_index[0]]
        for p in range(world):
            if p == rank:
                send_lists.append(torch.zeros(0, **i64))
                continue
            need = (dst_owner_all == p) & (src_owner_all == rank)
            ids = torch.unique(edge_index[0, need.nonzero(as_tuple=True)[0]])   # ascending = the peer's arrival order
            send_lists.append(owned_pos[ids])
        send_splits = [int(x.numel()) for x in send_lists]
        send_idx = torch.cat(send_lists) if send_lists else torch.zeros(0, **i64)
        active = torch.bincount(tkey[owned], minlength=num_types + 1).tolist()
        # processing order of the pull kernel: the k-th row of every owner, owners taken in the order rank+1, rank+2, ...
        # => consecutive work items cycle through all peers and no two ranks start on the same source
        lo_owner = owner[local_global]
        ordered = torch.argsort(lo_owner, stable=True)
        cnt = torch.bincount(lo_owner, minlength=world)
        start = torch.cumsum(cnt, 0) - cnt
        k_in_owner = torch.empty_like(lo_owner)
        k_in_owner[ordered] = torch.arange(lo_owner.numel(), device=wdev) - start[lo_owner[ordered]]
        pull_order = torch.argsort(k_in_owner * world + (lo_owner - rank - 1) % world, stable=True).to(torch.int32)
        # "auto" (default): fused peer-memory pull on CUDA, NCCL all_to_all if symmetric memory is unavailable
        mode = halo_mode or os.environ.get("HGT_HALO", "auto")
        return ShardedGraph(rank=rank, world=world, device=device, n_owned=n_owned, n_halo=n_halo,
                            n_local_edges=int(e_sel.numel()), owned_global=owned.cpu(), halo_global=halo.cpu(),
                            local_global=local_global.cpu(), node_type=node_type[local_global].to(device),
                            edge_index=ei_local.to(device), edge_type=edge_type[e_sel].to(device),
                            edge_time=None if edge_time is None else edge_time[e_sel].to(device),
                            send_idx=send_idx.to(device), send_splits=send_splits, recv_splits=recv_splits,
                            cat_index=order.to(torch.int32).to(device),
                            pull_rank=owner[local_global].to(torch.int32).to(device),
                            pull_row=owned_pos[local_global].to(torch.int32).to(device),
                            pull_order=pull_order.to(device),
                            own_rows=local_of[owned].to(device), active_per_type=active, max_owned=max_owned,
                            num_types=num_types, num_relations=num_relations, group=group, halo_mode=mode,
                            kv_runs=None if kv_runs is None else tuple(sorted(kv_runs.items())))

    # --------------------------------------------------------------------------------------------
    def _gather(self, src, idx32, n_rows):
        d = src.shape[1]
        if src.is_cuda:
            from . import _lib
            out = torch.empty((n_rows, d), dtype=src.dtype, device=src.device)
            if n_rows:
                _lib.call("hgt_gather_rows", src.contiguous().data_ptr(), idx32.data_ptr(), n_rows, d, out.data_ptr(),
                          torch.cuda.current_stream().cuda_stream)
            return out
        return src.index_select(0, idx32.long())

    def _resolve_halo_mode(self, x_own):
        """"auto" -> "p2p" or "nccl", decided ONCE and COLLECTIVELY: every rank tries the symmetric-memory rendezvous,
        the success flags are all-reduced (MIN) and the ranks switch together — a rank-local fallback would leave some
        ranks in NCCL's all_to_all and others in symmetric-memory barriers.  Only the rendezvous is guarded; kernel and
        ABI errors of the pull path propagate."""
        if self.halo_mode != "auto":
            return                                         # "nccl", "p2p" (pull) or "push" (experimental) chosen explicitly
        if not (x_own.is_cuda and self.world > 1):
            self.halo_mode = "nccl"
            return
        ok, why = 1, ""
        try:
            self._symm_setup(x_own.shape[1], x_own.device)
        except (RuntimeError, ImportError, AttributeError, NotImplementedError) as exc:   # symmetric memory unavailable
            ok, why = 0, str(exc)
        flag = torch.tensor([ok], dtype=torch.int32, device=x_own.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 1:
            self.halo_mode = "p2p"
        else:
            import warnings
            if why:
                warnings.warn("pyhgt_b200: symmetric-memory halo exchange unavailable on this rank (%s); all ranks use "
                              "the NCCL all_to_all" % why)
            self._symm = None
            self.halo_mode = "nccl"

    def exchange(self, x_own, split=False):
        """[n_owned, d] owned rows -> [n_local, d] local rows in local (type-sorted) order.  With split=True returns
        (x_local, (hi, lo) or None): on the p2p path the rows also come back as the bf16 hi/lo operand split and the fp32
        copy is valid for the owned rows only."""
        self._resolve_halo_mode(x_own)
        if self.halo_mode == "push" and x_own.is_cuda and self.world > 1 and split and x_own.shape[1] % 16 == 0 \
                and x_own.shape[1] >= 64:
            return self._exchange_push(x_own)
        if self.halo_mode in ("p2p", "push") and x_own.is_cuda and self.world > 1:
            return self._exchange_p2p(x_own, split)
        res = self._exchange_nccl(x_own)
        return (res, None) if split else res

    def halo_stats(self, d):
        """Bytes this rank receives per layer (fp32 halo rows) and the rows involved."""
        return {"halo_rows_rank": self.n_halo, "owned_rows_rank": self.n_owned,
                "halo_bytes_rank": self.n_halo * d * 4, "mode": self.halo_mode}

    def _exchange_nccl(self, x_own):
        d = x_own.shape[1]
        if getattr(self, "_send_idx32", None) is None:
            self._send_idx32 = self.send_idx.to(torch.int32)
        buf = torch.empty((self.n_owned + self.n_halo, d), dtype=x_own.dtype, device=x_own.device)
        buf[:self.n_owned].copy_(x_own)
        send = self._gather(x_own, self._send_idx32, self.send_idx.numel())
        if self.world > 1:
            dist.all_to_all_single(buf[self.n_owned:], send, self.recv_splits, self.send_splits, group=self.group)
        return self._gather(buf, self.cat_index, self.n_owned + self.n_halo)

    def _symm_setup(self, d, device):
        """One symmetric allocation holding TWO publish areas of max_owned rows each (used alternately)."""
        import torch.distributed._symmetric_memory as symm_mem
        if self._symm is None or self._symm[0].shape[1] != d:
            buf = symm_mem.empty((2 * max(self.max_owned, 1), d), dtype=torch.float32, device=device)
            hdl = symm_mem.rendezvous(buf, self.group if self.group is not None else dist.group.WORLD)
            self._symm = (buf, hdl)
            self._slot = 0
        return self._symm

    def input_buffer(self, d, slot=0):
        """[n_owned, d] view of publish area `slot` (0 / 1) in NVLink-mapped symmetric memory: a layer input that lives
        here needs no publish copy — `forward` recognises it.  A producer alternates the slots from layer to layer (the
        one barrier of an exchange then also covers the write-after-read hazard).  Plain tensor when the exchange goes
        through NCCL."""
        dev = self.device if isinstance(self.device, torch.device) else torch.device(self.device)
        probe = torch.empty((0, d), dtype=torch.float32, device=dev)
        self._resolve_halo_mode(probe)
        if self.halo_mode != "p2p":
            return torch.empty((self.n_owned, d), dtype=torch.float32, device=dev)
        buf, _ = self._symm_setup(d, dev)
        m = max(self.max_owned, 1)
        return buf[slot * m:slot * m + self.n_owned]

    def _exchange_p2p(self, x_own, split=False):
        """Fused halo exchange: every rank publishes x_own in NVLink-mapped symmetric memory and ONE kernel pulls
        each local row (owned and halo alike) straight from its owner's HBM into type-sorted position — no send-side
        gather, no NCCL call, no re-ordering pass.  Two publish areas are used alternately, so ONE barrier per
        exchange is enough: it says "everybody's rows are published" and, because every rank reaches it only after
        its previous pull, also "nobody still reads the area written next"."""
        from . import _lib
        d = x_own.shape[1]
        buf, hdl = self._symm_setup(d, x_own.device)
        m = max(self.max_owned, 1)
        slot = -1
        for k in (0, 1):
            if x_own.data_ptr() == buf[k * m:].data_ptr() and x_own.is_contiguous():
                slot = k                                 # already published in place (input_buffer)
        if slot < 0:
            slot = self._slot
            buf[slot * m:slot * m + self.n_owned].copy_(x_own)
        self._slot = slot ^ 1
        hdl.barrier(channel=0)                       # every rank's rows are published (and the other area is free)
        n_local = self.n_owned + self.n_halo
        x_local = torch.empty((n_local, d), dtype=torch.float32, device=x_own.device)
        if split and d % 16 == 0 and d >= 64:
            # fused pull + bf16 hi/lo conversion: halo rows never exist in fp32 on this rank
            hi = torch.empty((n_local, d), dtype=torch.bfloat16, device=x_own.device)
            lo = torch.empty((n_local, d), dtype=torch.bfloat16, device=x_own.device)
            from .conv import HGTConv
            with HGTConv._stage("halo_pull_kernel"):               # bench.py: the kernel alone, without barrier / publish
                _lib.call("hgt_halo_pull_split", hdl.buffer_ptrs_dev, self.pull_rank.data_ptr(),
                          self.pull_row.data_ptr(), _lib.ptr(self.pull_order), n_local, d, self.rank, slot * m,
                          x_local.data_ptr(), hi.data_ptr(), lo.data_ptr(), torch.cuda.current_stream().cuda_stream)
            return x_local, (hi, lo)
        _lib.call("hgt_halo_pull", hdl.buffer_ptrs_dev, self.pull_rank.data_ptr(), self.pull_row.data_ptr(), n_local, d,
                  slot * m, x_local.data_ptr(), torch.cuda.current_stream().cuda_stream)
        return (x_local, None) if split else x_local

    # ---- push variant (experimental, opt-in with halo_mode="push") -------------------------------------------------
    def _push_setup(self, d, device):
        """Collective, once: turn every rank's pull plan into the owners' push plans (one all-to-all of (row, destination
        row) pairs) and allocate the symmetric destination buffers (two areas of max_local rows for hi and for lo)."""
        import torch.distributed._symmetric_memory as symm_mem
        if getattr(self, "_push", None) is not None and self._push["d"] == d:
            return self._push
        W, grp = self.world, (self.group if self.group is not None else dist.group.WORLD)
        n_local = self.n_owned + self.n_halo
        pr = self.pull_rank.long()
        cnt_from = torch.bincount(pr, minlength=W)
        cnt_to = torch.empty_like(cnt_from)
        dist.all_to_all_single(cnt_to, cnt_from, group=grp)
        order = torch.argsort(pr, stable=True)                              # my local rows grouped by their owner
        send = torch.stack([self.pull_row.long()[order], order], 1).contiguous()
        recv = torch.empty((int(cnt_to.sum()), 2), dtype=torch.int64, device=device)
        dist.all_to_all_single(recv, send, output_split_sizes=cnt_to.tolist(), input_split_sizes=cnt_from.tolist(),
                               group=grp)
        peer = torch.repeat_interleave(torch.arange(W, device=device), cnt_to)
        # item order: the k-th item of every consumer, consumers taken from rank+1 round the ring (same idea as pull_order)
        start = torch.cumsum(cnt_to, 0) - cnt_to
        k_in = torch.arange(peer.numel(), device=device) - start[peer]
        o = torch.argsort(k_in * W + (peer - self.rank - 1) % W, stable=True)
        mx = torch.tensor([n_local], dtype=torch.int64, device=device)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=grp)
        max_local = int(mx.item())
        hi = symm_mem.empty((2 * max_local, d), dtype=torch.bfloat16, device=device)
        lo = symm_mem.empty((2 * max_local, d), dtype=torch.bfloat16, device=device)
        h_hi, h_lo = symm_mem.rendezvous(hi, grp), symm_mem.rendezvous(lo, grp)
        self._push = dict(d=d, peer=peer[o].to(torch.int32), src=recv[o, 0].to(torch.int32), dst=recv[o, 1].to(torch.int32),
                          hi=hi, lo=lo, h_hi=h_hi, h_lo=h_lo, max_local=max_local, slot=0)
        return self._push

    def _exchange_push(self, x_own):
        """Owners push: one kernel converts my owned rows and stores their bf16 hi/lo split into every consumer's operand
        buffers (and into mine); ONE barrier, then the projection reads its operands in place."""
        from . import _lib
        from .conv import HGTConv
        d = x_own.shape[1]
        P = self._push_setup(d, x_own.device)
        slot = P["slot"]
        P["slot"] = slot ^ 1
        n_local = self.n_owned + self.n_halo
        x_local = torch.empty((n_local, d), dtype=torch.float32, device=x_own.device)   # valid for the owned rows only
        xo = x_own.contiguous()
        with HGTConv._stage("halo_push_kernel"):
            _lib.call("hgt_halo_push_split", xo.data_ptr(), P["peer"].data_ptr(), P["src"].data_ptr(), P["dst"].data_ptr(),
                      P["peer"].numel(), d, self.rank, slot * P["max_local"], P["h_hi"].buffer_ptrs_dev,
                      P["h_lo"].buffer_ptrs_dev, x_local.data_ptr(), torch.cuda.current_stream().cuda_stream)
        P["h_hi"].barrier(channel=0)                  # every owner's stores have landed (and the other area is free again)
        base = slot * P["max_local"]
        return x_local, (P["hi"][base:base + n_local], P["lo"][base:base + n_local])

    def forward_train(self, conv, x_own):
        """Differentiable sharded layer (BASELINE config 4): halo exchange with a reverse all-to-all in backward, the
        layer's autograd path on the local graph, owned rows out.  Parameter gradients are PARTIAL per rank (each rank
        sees only its destinations): sum them with `allreduce_grads` (or wrap the model in DistributedDataParallel)."""
        _require_fp32_kv(conv)
        x_local = _HaloExchange.apply(x_own, self)
        tm = self.edge_time if conv.use_RTE else None
        if x_local.is_cuda and hasattr(conv, "q_linears") and type(conv).__name__ == "HGTConv":
            # only the owned prefix of every type is a destination here: Q / a_linear / update skip the halo rows
            from .autograd import hgt_conv_autograd
            conv._check_inputs(x_local, tm)
            out = hgt_conv_autograd(conv, x_local, self.node_type, self.edge_index, self.edge_type, tm,
                                    active=self.active_per_type, kv_runs=self.kv_runs)
        else:
            out = conv(x_local, self.node_type, self.edge_index, self.edge_type, tm)
        return out.index_select(0, self.own_rows)

    def allreduce_grads(self, module):
        if self.world > 1:
            for p in module.parameters():
                if p.grad is not None:
                    dist.all_reduce(p.grad, group=self.group)

    def forward(self, conv, x_own, graph=None):
        """One HGTConv layer on this rank's shard; returns the [n_owned, d] output rows (owned_global order).
        `graph` = (node_type, edge_index, edge_type, edge_time) device tensors holding this rank's LOCAL graph, for
        callers that stream the shard from the host every step (the plan is rebuilt when they change)."""
        from .conv import HGTConv
        _require_fp32_kv(conv)
        with HGTConv._stage("halo_exchange"):
            x_local, x_split = self.exchange(x_own, split=x_own.is_cuda and conv.linear_impl in (0, 2))
        l_nt, l_ei, l_et, l_tm = (self.node_type, self.edge_index, self.edge_type, self.edge_time) if graph is None else graph
        if x_local.is_cuda:
            # the update epilogue writes each owned row straight to its position in owned_global order
            if getattr(self, "_out_map", None) is None:
                om = torch.full((self.n_owned + self.n_halo,), -1, dtype=torch.int32, device=x_local.device)
                om[self.own_rows] = torch.arange(self.n_owned, dtype=torch.int32, device=x_local.device)
                self._out_map = om
            out, att, _ = conv._forward_impl(x_local, l_nt, l_ei, l_et,
                                             l_tm if conv.use_RTE else None, want_att=False, save=False,
                                             active_per_type=self.active_per_type, out_map=self._out_map,
                                             out_rows=self.n_owned, x_split=x_split, kv_runs=self.kv_runs)
            return out
        out, att, _ = conv._forward_impl(x_local, l_nt, l_ei, l_et,
                                         l_tm if conv.use_RTE else None, want_att=False, save=False,
                                         active_per_type=self.active_per_type)
        return out.index_select(0, self.own_rows)
