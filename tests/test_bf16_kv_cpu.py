"""CPU checks of the bf16 K'/V' inference mode (HGTConv.kv_dtype): the fp64 emulation of its contract
(tests/bf16_kv_oracle.py), the C-ABI declarations and bindings, and the Python switch."""
import copy
import ctypes
import io
import os
import pickle
import re

import pytest
import torch

from oracle import hgt_oracle
from tests.bf16_kv_oracle import hgt_forward_bf16kv_fp64, rel_fro
from tests.conftest import CONV_FIXTURES, ROOT, load_golden

# Relative Frobenius distance of the emulated bf16 layer from the fp64 layer on every golden (measured:
# c1_norte 3.95e-4, c1_rte 4.39e-4, rand_t3r4_dk4 2.99e-4, rand_dk25 6.18e-4, mag_mini_dk50 1.79e-4, oag_mini 3.80e-4,
# hub_h2 5.88e-4).  The upper bounds carry a 1.5x margin; the lower bound shows that the rounding is really applied.
EMU_FRO_MAX = {"c1_norte": 6.0e-4, "c1_rte": 6.6e-4, "rand_t3r4_dk4": 4.5e-4, "rand_dk25": 9.3e-4,
               "mag_mini_dk50": 2.7e-4, "oag_mini": 5.7e-4, "hub_h2": 8.8e-4}
EMU_FRO_MIN = 5e-5
EMU_MAXABS_MAX = 1e-2


def _args(fx):
    c = fx["cfg"]
    kw = dict(num_types=c["num_types"], num_relations=c["num_relations"], n_heads=c["n_heads"],
              use_norm=c["use_norm"], use_RTE=c["use_RTE"])
    return (fx["state_dict"], fx["node_inp"], fx["node_type"], fx["edge_index"], fx["edge_type"], fx["edge_time"]), kw


@pytest.mark.parametrize("name", CONV_FIXTURES)
def test_emulation_without_rounding_is_the_fp64_layer(name):
    a, kw = _args(load_golden(name))
    ref, ref_att = hgt_oracle.hgt_forward_dense_fp64(*a, **kw)
    out, att = hgt_forward_bf16kv_fp64(*a, round_kv=False, **kw)
    assert (out - ref).abs().max().item() <= 1e-12
    assert (att - ref_att).abs().max().item() <= 1e-12


@pytest.mark.parametrize("name", CONV_FIXTURES)
def test_emulation_distance_from_fp64_is_bounded(name):
    a, kw = _args(load_golden(name))
    ref, _ = hgt_oracle.hgt_forward_dense_fp64(*a, **kw)
    out, _ = hgt_forward_bf16kv_fp64(*a, **kw)
    fro = rel_fro(out, ref)
    assert EMU_FRO_MIN <= fro <= EMU_FRO_MAX[name], "%s: rel Frobenius %.3e" % (name, fro)
    assert (out - ref).abs().max().item() <= EMU_MAXABS_MAX


def test_emulation_rounds_rows_to_nearest_even():
    """The rounding helper is torch's fp32 -> bf16 conversion (round to nearest, ties to even)."""
    from tests.bf16_kv_oracle import _rnd
    x = torch.tensor([1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8, -(1.0 + 2 ** -8), 1.0 + 2 ** -8 + 2 ** -20], dtype=torch.float64)
    assert _rnd(x).tolist() == [1.0, 1.0 + 2 ** -6, -1.0, 1.0 + 2 ** -7]


def _declared():
    text = open(os.path.join(ROOT, "include", "hgt_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return set(re.findall(r"\b(hgt_[a-z0-9_]+)\s*\(", text))


NEW_SYMBOLS = ["hgt_typed_linear_bf16", "hgt_typed_linear_bf16_workspace_bytes", "hgt_typed_linear_presplit_bf16",
               "hgt_typed_linear_presplit_bf16_workspace_bytes", "hgt_edge_forward_bf16kv"]


def test_bf16_entry_points_are_declared_bound_and_exported():
    from pyhgt_b200 import _lib
    lib = _lib.load()
    for name in NEW_SYMBOLS:
        assert name in _declared(), name
        assert name in _lib.SIGNATURES, name
        assert hasattr(lib, name), name
    # same arguments as the fp32 siblings (pointer types aside)
    assert _lib.SIGNATURES["hgt_typed_linear_bf16"] == _lib.SIGNATURES["hgt_typed_linear"]
    assert _lib.SIGNATURES["hgt_typed_linear_presplit_bf16"] == _lib.SIGNATURES["hgt_typed_linear_presplit"]
    assert _lib.SIGNATURES["hgt_edge_forward_bf16kv"] == _lib.SIGNATURES["hgt_edge_forward"]


def test_conv_args_end_with_the_bf16_fields():
    from pyhgt_b200 import _lib
    lib = _lib.load()
    assert ctypes.sizeof(_lib.ConvArgs) == lib.hgt_conv_args_size()
    names = [f[0] for f in _lib.ConvArgs._fields_]
    assert names[-2:] == ["kv_bf16", "n_q_groups"]
    assert _lib.ConvArgs.kv_bf16.offset > _lib.ConvArgs.out_lo.offset
    assert _lib.ConvArgs().kv_bf16 == 0                      # a zero-initialised block is the fp32 layer


def test_set_kv_dtype_walks_the_module_tree():
    import pyhgt_b200
    from pyhgt_b200.model import GNN
    g = GNN(in_dim=32, n_hid=64, num_types=3, num_relations=2, n_heads=4, n_layers=3)
    sd = {k: v.clone() for k, v in g.state_dict().items()}
    assert pyhgt_b200.set_kv_dtype(g, torch.bfloat16) is g
    convs = [gc.base_conv for gc in g.gcs]
    assert all(c.kv_dtype == torch.bfloat16 for c in convs)
    assert pyhgt_b200.HGTConv.kv_dtype == torch.float32        # the class default is untouched
    assert list(g.state_dict()) == list(sd)
    buf = io.BytesIO()
    torch.save(g, buf)
    buf.seek(0)
    g2 = torch.load(buf, weights_only=False)
    assert all(gc.base_conv.kv_dtype == torch.bfloat16 for gc in g2.gcs)
    assert pickle.loads(pickle.dumps(convs[0])).kv_dtype == torch.bfloat16
    assert copy.deepcopy(convs[0]).kv_dtype == torch.bfloat16
    pyhgt_b200.set_kv_dtype(g, torch.float32)
    assert all("kv_dtype" in c.__dict__ and c.kv_dtype == torch.float32 for c in convs)


def test_set_kv_dtype_rejects_other_dtypes():
    import pyhgt_b200
    m = pyhgt_b200.HGTConv(16, 16, 2, 1, 2)
    for dt in (torch.float16, torch.float64, "bfloat16"):
        with pytest.raises(ValueError):
            pyhgt_b200.set_kv_dtype(m, dt)
    m.kv_dtype = torch.float16
    with pytest.raises(ValueError, match="kv_dtype"):
        m._kv_bf16()
    d = pyhgt_b200.DenseHGTConv(16, 16, 2, 1, 2)
    d.kv_dtype = torch.bfloat16
    with pytest.raises(ValueError, match="DenseHGTConv"):
        d._kv_bf16()
