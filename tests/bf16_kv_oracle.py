"""fp64 emulation of HGTConv's bf16 K'/V' inference mode (HGTConv.kv_dtype = torch.bfloat16).  TEST INFRASTRUCTURE ONLY.

The mode's contract: the layer is the fp32 pipeline with one change, every row of the folded [K'|V'] table and of the
RTE tables K'R/V'R is rounded to bf16 (round to nearest even) after its GEMM, bias included.  This restatement computes
everything in float64 and rounds exactly those rows (through fp32, as the GPU rounds its fp32 GEMM result), so it
isolates the effect of the rounding from that of fp32 arithmetic:

    K'[j,p] = pri[r] / sqrt(d_k) * att[r]^T (W_k^s x_j + b_k^s)        V'[j,p] = msg[r]^T (W_v^s x_j + b_v^s)
    K'R[p,dt] = pri[r] / sqrt(d_k) * att[r]^T W_k^s RT[dt]              V'R[p,dt] = msg[r]^T W_v^s RT[dt]
    per edge j -r-> i at time dt:  k = bf16(K'[j,p]) + bf16(K'R[p,dt]),  v = bf16(V'[j,p]) + bf16(V'R[p,dt])

with p = <type(j), r>.  With round_kv=False it is an independent regrouping of oracle.hgt_oracle.hgt_forward_dense_fp64
(relation_pri folded into K', the RTE term projected separately) and agrees with it to rounding error.
"""
import math

import torch
import torch.nn.functional as F


def _rnd(t):
    return t.float().bfloat16().double()


def hgt_forward_bf16kv_fp64(params, node_inp, node_type, edge_index, edge_type, edge_time=None, *, num_types,
                            num_relations, n_heads, use_norm=True, use_RTE=True, round_kv=True):
    """Returns (out [N,d], att [E,H]) in float64."""
    p = {k: v.double() for k, v in params.items()}
    x = node_inp.double()
    n_nodes = x.shape[0]
    d = p["q_linears.0.weight"].shape[0]
    d_k = d // n_heads
    src, dst = edge_index[0], edge_index[1]
    n_edges = src.numel()
    valid_t = (node_type >= 0) & (node_type < num_types)
    tt = node_type.clamp(0, num_types - 1)
    rnd = _rnd if round_kv else (lambda t: t)

    def stack(name, part):
        return torch.stack([p["%s.%d.%s" % (name, t, part)] for t in range(num_types)])

    def typed(name, inp):
        return torch.einsum("ni,noi->no", inp, stack(name, "weight")[tt]) + stack(name, "bias")[tt]

    q_all = typed("q_linears", x)
    rr = edge_type.clamp(0, num_relations - 1)
    ts = tt[src]
    scale = (p["relation_pri"][rr] / math.sqrt(d_k))[:, :, None]                       # [E, H, 1]

    def fold_k(rows):                                                                  # [E, d] -> folded K' rows
        return torch.einsum("eha,ehab->ehb", rows.view(-1, n_heads, d_k), p["relation_att"][rr]) * scale

    def fold_v(rows):
        return torch.einsum("eha,ehab->ehb", rows.view(-1, n_heads, d_k), p["relation_msg"][rr])

    k_e = rnd(fold_k(typed("k_linears", x)[src]))
    v_e = rnd(fold_v(typed("v_linears", x)[src]))
    if use_RTE:
        rt = p["emb.emb.weight"] @ p["emb.lin.weight"].t() + p["emb.lin.bias"]         # [240, d]
        rt_e = rt[edge_time]
        k_e = k_e + rnd(fold_k(torch.einsum("ei,eoi->eo", rt_e, stack("k_linears", "weight")[ts])))
        v_e = v_e + rnd(fold_v(torch.einsum("ei,eoi->eo", rt_e, stack("v_linears", "weight")[ts])))
    ok = valid_t[src] & valid_t[dst] & (edge_type >= 0) & (edge_type < num_relations)
    s = (q_all[dst].view(-1, n_heads, d_k) * k_e).sum(-1)
    s = torch.where(ok[:, None], s, torch.zeros_like(s))             # edges matching no triple: score 0, message 0
    v_e = torch.where(ok[:, None, None], v_e, torch.zeros_like(v_e))
    att = torch.zeros(n_edges, n_heads, dtype=torch.float64)
    agg = torch.zeros(n_nodes, n_heads, d_k, dtype=torch.float64)
    order = torch.argsort(dst, stable=True)
    counts = torch.bincount(dst, minlength=n_nodes)
    start = 0
    for n in range(n_nodes):
        c = int(counts[n])
        if c == 0:
            continue
        e = order[start:start + c]
        start += c
        sc = s[e]
        pr = torch.exp(sc - sc.max(0, keepdim=True).values)
        pr = pr / (pr.sum(0, keepdim=True) + 1e-16)
        att[e] = pr
        agg[n] = (pr[:, :, None] * v_e[e]).sum(0)
    g = F.gelu(agg.view(n_nodes, d))
    out = torch.zeros(n_nodes, d, dtype=torch.float64)
    for t in range(num_types):
        sel = node_type == t
        if int(sel.sum()) == 0:
            continue
        o = g[sel] @ p["a_linears.%d.weight" % t].t() + p["a_linears.%d.bias" % t]
        a = torch.sigmoid(p["skip"][t])
        y = o * a + x[sel] * (1 - a)
        if use_norm:
            y = F.layer_norm(y, (d,), p["norms.%d.weight" % t], p["norms.%d.bias" % t], 1e-5)
        out[sel] = y
    return out, att


def rel_fro(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))
