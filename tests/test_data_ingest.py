"""pyhgt_b200.data.to_torch (SURVEY.md §8f rank 2) against the reference's own to_torch (pyHGT/data.py:212-256):
the golden fixture was produced by the unmodified reference on a synthetic sampled sub-graph (oracle/make_golden.py);
outputs must be IDENTICAL (node order, edge order, dtypes, dict contents)."""
import torch

from pyhgt_b200 import data as hdata
from tests.conftest import load_golden, load_record


class _GraphStub:
    """What to_torch needs from the reference's Graph: get_types() and get_meta_graph()."""

    def __init__(self, types, metas):
        self._t, self._m = list(types), [tuple(m) for m in metas]

    def get_types(self):
        return self._t

    def get_meta_graph(self):
        return self._m


def test_to_torch_is_identical_to_reference_golden():
    fx = load_golden("to_torch")
    g = _GraphStub(fx["types"], fx["meta_graph"])
    out = hdata.to_torch(fx["feature"], fx["time"], fx["edge_list"], g)
    for got, key in zip(out[:5], ("node_feature", "node_type", "edge_time", "edge_index", "edge_type")):
        ref = fx[key]
        assert got.dtype == ref.dtype and got.shape == ref.shape, key
        assert torch.equal(got, ref), key
    assert out[5] == fx["node_dict"] and out[6] == fx["edge_dict"]
    assert out[3].dtype == torch.int64 and out[0].dtype == torch.float32


def test_to_torch_empty_edge_list():
    fx = load_golden("to_torch")
    g = _GraphStub(fx["types"], fx["meta_graph"])
    out = hdata.to_torch(fx["feature"], fx["time"], {}, g)
    assert out[3].shape == (2, 0) and out[4].numel() == 0 and out[2].numel() == 0
    assert torch.equal(out[0], fx["node_feature"])


def test_to_torch_matches_reference_on_a_larger_graph():
    """5,300 nodes / 65,300 edges: digests of the reference's tensors and its node / edge dicts, recorded in
    tests/golden/reference_record.json (oracle/make_golden.py:reference_record)."""
    from oracle import make_golden as mg
    rec = load_record()["to_torch_large"]
    fx = load_golden("to_torch")                                # the reference's type order and meta graph
    feature, times, edge_list = mg.sampled_subgraph_inputs(rec["seed"], fx["types"], fx["meta_graph"],
                                                          rec["n_per_type"], rec["n_edges"])
    out = hdata.to_torch(feature, times, edge_list, _GraphStub(fx["types"], fx["meta_graph"]))
    for got, key in zip(out[:5], ("node_feature", "node_type", "edge_time", "edge_index", "edge_type")):
        assert mg.digest(got) == rec[key], key
    assert out[5] == rec["node_dict"] and out[6] == rec["edge_dict"]
