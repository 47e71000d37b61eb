"""Drop-in contract of pyhgt_b200.HGTConv on the host side (no GPU): constructor, attributes, parameter
names/shapes (state_dict compatibility with reference checkpoints), repr.  Reference: conv.py:12-54,136-139."""
import math

import pytest
import torch

import pyhgt_b200
from tests.conftest import load_golden, load_record


def test_param_count_known_answer():
    # one MAG-recipe layer = 5,182,028 parameters (4 layers + adapters + classifier = 21,173,389,
    # ogbn-mag/README.md:30)
    m = pyhgt_b200.HGTConv(512, 512, 4, 9, 8, 0.2, True, True)
    assert sum(p.numel() for p in m.parameters()) == 5182028


def test_state_dict_loads_reference_checkpoint(conv_fixture):
    c = conv_fixture["cfg"]
    m = pyhgt_b200.HGTConv(c["in_dim"], c["out_dim"], c["num_types"], c["num_relations"], c["n_heads"], 0.2,
                           c["use_norm"], c["use_RTE"])
    sd = conv_fixture["state_dict"]
    assert list(m.state_dict().keys()) == list(sd.keys())
    for k, v in m.state_dict().items():
        assert tuple(v.shape) == tuple(sd[k].shape), k
    m.load_state_dict(sd, strict=True)


def test_public_attributes_and_repr():
    m = pyhgt_b200.HGTConv(64, 64, 3, 5, 4, 0.1, False, False)
    assert (m.in_dim, m.out_dim, m.num_types, m.num_relations, m.n_heads, m.d_k) == (64, 64, 3, 5, 4, 16)
    assert m.total_rel == 3 * 5 * 3 and m.sqrt_dk == math.sqrt(16) and m.att is None
    assert m.use_norm is False and m.use_RTE is False and not hasattr(m, "emb") and len(m.norms) == 0
    assert repr(m) == "HGTConv(in_dim=64, out_dim=64, num_types=3, num_types=5)"   # (sic) conv.py:137
    assert torch.all(m.relation_pri == 1) and torch.all(m.skip == 1)
    a = math.sqrt(6.0 / 32)
    assert m.relation_att.abs().max() <= a and m.relation_msg.abs().max() <= a


def test_rte_table_matches_oracle_formula():
    from oracle import hgt_oracle
    m = pyhgt_b200.RelTemporalEncoding(64)
    assert torch.allclose(m.emb.weight.detach(), hgt_oracle.rte_sinusoid_table(64))
    assert m.emb.weight.requires_grad          # the reference leaves the table trainable (SURVEY §8 a8)


def test_parameter_names_equal_reference_module():
    ref = load_record()["hgtconv_32_3_4_4_params"]          # the reference's HGTConv(32, 32, 3, 4, 4, 0.2, True, True)
    mine = pyhgt_b200.HGTConv(32, 32, 3, 4, 4, 0.2, True, True)
    assert [(n, tuple(s)) for n, s in ref] == [(n, tuple(p.shape)) for n, p in mine.named_parameters()]


def test_general_conv_dispatch():
    g = pyhgt_b200.GeneralConv('hgt', 32, 32, 2, 3, 4, 0.2, True, False)
    assert isinstance(g.base_conv, pyhgt_b200.HGTConv) and g.base_conv.use_RTE is False
    d = pyhgt_b200.GeneralConv('dense_hgt', 32, 32, 2, 3, 4, 0.2, True, True)
    assert isinstance(d.base_conv, pyhgt_b200.DenseHGTConv) and not hasattr(d.base_conv, "skip")
    with pytest.raises(NotImplementedError):
        pyhgt_b200.GeneralConv('gcn', 32, 32, 2, 3, 4, 0.2)


def test_dense_hgt_state_dict_matches_reference_fixture():
    fx = load_golden("dense_hgt")
    c = fx["cfg"]
    m = pyhgt_b200.DenseHGTConv(c["in_dim"], c["out_dim"], c["num_types"], c["num_relations"], c["n_heads"], 0.2,
                                c["use_norm"], c["use_RTE"])
    assert list(m.state_dict().keys()) == list(fx["state_dict"].keys())
    m.load_state_dict(fx["state_dict"], strict=True)


def test_gnn_wrapper_state_dict_matches_reference_fixture():
    from pyhgt_b200.model import GNN
    fx = load_golden("gnn_2layer")
    c = fx["cfg"]
    m = GNN(c["in_dim"], c["n_hid"], c["num_types"], c["num_relations"], c["n_heads"], c["n_layers"], 0.2, "hgt",
            c["prev_norm"], c["last_norm"], c["use_RTE"])
    assert list(m.state_dict().keys()) == list(fx["state_dict"].keys())
    m.load_state_dict(fx["state_dict"], strict=True)


def test_module_pickles_and_deep_copies_with_launch_caches():
    """OAG/train_paper_field.py:279 `torch.save(model, ...)` right after an eval pass: the per-process launch caches
    (ctypes argument blocks, pointer tables) must not travel with the module."""
    import copy
    import io
    import pyhgt_b200
    from pyhgt_b200 import _lib
    m = pyhgt_b200.HGTConv(64, 64, 2, 1, 4)
    m.__dict__["_args_cache"] = {("k",): (_lib.ConvArgs(), None, None, None)}     # what _forward_fused leaves behind
    m._ptrs("wq", [l.weight for l in m.q_linears], torch.device("cpu"))
    m2 = copy.deepcopy(m)
    buf = io.BytesIO()
    torch.save(m, buf)
    buf.seek(0)
    m3 = torch.load(buf, weights_only=False)
    for other in (m2, m3):
        assert "_args_cache" not in other.__dict__ and other._ptr_tables == {}
        for (k, a), (k2, b) in zip(m.state_dict().items(), other.state_dict().items()):
            assert k == k2 and torch.equal(a, b)
    assert "_args_cache" in m.__dict__                                            # the live module keeps its caches
