"""Pin the CPU oracle (oracle/hgt_oracle.py) against outputs of the reference itself:
tests/golden/*.pt were produced by /root/reference/pyHGT/conv.py (oracle/make_golden.py)."""
import math

import pytest
import torch

from oracle import hgt_oracle
from tests.conftest import load_record


def _kw(fx):
    c = fx["cfg"]
    return dict(num_types=c["num_types"], num_relations=c["num_relations"], n_heads=c["n_heads"],
                use_norm=c["use_norm"], use_RTE=c["use_RTE"])


def test_ref_port_matches_reference_golden(conv_fixture):
    fx = conv_fixture
    out, att = hgt_oracle.hgt_forward_ref_port(fx["state_dict"], fx["node_inp"], fx["node_type"],
                                               fx["edge_index"], fx["edge_type"], fx["edge_time"], **_kw(fx))
    # same fp32 ops in the same order as the reference: expect (near) bit equality
    assert torch.allclose(out, fx["out"], rtol=1e-6, atol=1e-6)
    assert torch.allclose(att, fx["att"], rtol=1e-6, atol=1e-7)


def test_dense_fp64_matches_reference_golden(conv_fixture):
    fx = conv_fixture
    out, att = hgt_oracle.hgt_forward_dense_fp64(fx["state_dict"], fx["node_inp"], fx["node_type"],
                                                 fx["edge_index"], fx["edge_type"], fx["edge_time"], **_kw(fx))
    assert torch.allclose(out.float(), fx["out"], rtol=2e-4, atol=2e-4)
    assert torch.allclose(att.float(), fx["att"], rtol=2e-4, atol=1e-5)


def test_softmax_rows_sum_to_one(conv_fixture):
    fx = conv_fixture
    dst = fx["edge_index"][1]
    n = fx["node_inp"].shape[0]
    sums = torch.zeros(n, fx["att"].shape[1]).index_add_(0, dst, fx["att"])
    has_in = torch.bincount(dst, minlength=n) > 0
    assert torch.allclose(sums[has_in], torch.ones_like(sums[has_in]), atol=1e-5)
    assert torch.all(sums[~has_in] == 0)


def test_init_params_inventory_matches_reference_count():
    """Known-answer: one MAG-recipe HGTConv has 5,182,028 parameters (SURVEY.md §4; the full model's
    21,173,389 is quoted at ogbn-mag/README.md:30)."""
    p = hgt_oracle.init_params(512, 512, 4, 9, 8, use_norm=True, use_RTE=True)
    assert sum(v.numel() for v in p.values()) == 5182028


def test_reference_model_param_count_known_answer():
    """The reference's MAG model (GNN + Classifier, inventories in tests/golden/reference_record.json) has 21,173,389
    parameters, and pyhgt_b200's GNN of the same shape has the reference GNN's parameter names and shapes."""
    from pyhgt_b200.model import GNN
    rec = load_record()
    g, c = rec["mag_gnn_params"], rec["mag_classifier_params"]
    assert sum(math.prod(s) for _, s in g) + sum(math.prod(s) for _, s in c) == 21173389
    mine = GNN(in_dim=129, n_hid=512, num_types=4, num_relations=9, n_heads=8, n_layers=4,
               prev_norm=True, last_norm=True, use_RTE=True)
    assert [(n, tuple(p.shape)) for n, p in mine.named_parameters()] == [(n, tuple(s)) for n, s in g]


def _random_case(seed, n=120, e=900, T=3, R=4, d=16, H=4, rte=True):
    from pyhgt_b200 import synth
    g = synth.make_random(n, e, T, R, seed=seed, isolated_frac=0.2, self_loops=10, duplicate_edges=20)
    params = hgt_oracle.init_params(d, d, T, R, H, use_norm=True, use_RTE=rte, seed=seed + 1)
    gen = torch.Generator().manual_seed(seed + 2)
    for k in list(params):                                  # move the constant inits (skip, pri, LayerNorm) off 1 / 0
        if k in ("skip", "relation_pri") or k.startswith("norms"):
            params[k] = params[k] + 0.3 * torch.randn(params[k].shape, generator=gen)
    x = torch.randn(g.num_nodes, d, generator=gen)
    kw = dict(num_types=T, num_relations=R, n_heads=H, use_norm=True, use_RTE=rte)
    return g, params, x, kw


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_port_and_dense_fp64_agree_on_random_graphs(seed):
    """The two independent restatements (per-triple fp32 port, node-level fp64) agree beyond the fixtures."""
    g, params, x, kw = _random_case(seed, rte=bool(seed % 2))
    o1, a1 = hgt_oracle.hgt_forward_ref_port(params, x, g.node_type, g.edge_index, g.edge_type, g.edge_time, **kw)
    o2, a2 = hgt_oracle.hgt_forward_dense_fp64(params, x, g.node_type, g.edge_index, g.edge_type, g.edge_time, **kw)
    assert torch.allclose(o1, o2.float(), rtol=2e-4, atol=2e-4)
    assert torch.allclose(a1, a2.float(), rtol=2e-4, atol=1e-5)


def test_oracle_invariances():
    """Permuting the edge list permutes att and leaves out unchanged; relabelling the nodes permutes out rows."""
    g, params, x, kw = _random_case(7)
    out, att = hgt_oracle.hgt_forward_ref_port(params, x, g.node_type, g.edge_index, g.edge_type, g.edge_time, **kw)
    gen = torch.Generator().manual_seed(0)
    pe = torch.randperm(g.num_edges, generator=gen)
    out2, att2 = hgt_oracle.hgt_forward_ref_port(params, x, g.node_type, g.edge_index[:, pe], g.edge_type[pe],
                                                 g.edge_time[pe], **kw)
    assert torch.allclose(out2, out, atol=1e-5) and torch.allclose(att2, att[pe], atol=1e-6)
    pn = torch.randperm(g.num_nodes, generator=gen)        # new id of old node i is inv[i]
    inv = torch.empty_like(pn); inv[pn] = torch.arange(g.num_nodes)
    out3, _ = hgt_oracle.hgt_forward_ref_port(params, x[pn], g.node_type[pn], inv[g.edge_index], g.edge_type,
                                              g.edge_time, **kw)
    assert torch.allclose(out3, out[pn], atol=1e-5)
