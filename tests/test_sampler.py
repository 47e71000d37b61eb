"""pyhgt_b200.sampler.sample_subgraph (SURVEY.md §8f rank 4) against the reference's own HGSampling
(pyHGT/data.py:87-210): with the same numpy seed the outputs are IDENTICAL — sampled nodes and their order, edge blocks
and their order, the tensors `to_torch` builds from them — and the global RNG ends in the same state (the same number of
draws was consumed).  The golden fixture was produced by the unmodified reference (oracle/make_golden.py:sampler_case)."""
import types

import numpy as np
import pytest
import torch

from pyhgt_b200 import data as hdata, sampler
from tests.conftest import load_golden, load_record


def _extractor(layer_data, graph):
    feature, times, indxs = {}, {}, {}
    for _type in layer_data:
        if len(layer_data[_type]) == 0:
            continue
        idxs = np.array(list(layer_data[_type].keys()))
        tims = np.array(list(layer_data[_type].values()))[:, 1]
        feature[_type] = np.stack([idxs, tims], 1).astype(np.float32)
        times[_type] = tims
        indxs[_type] = idxs
    return feature, times, indxs, []


def _norm(edge_list):
    return [(t, s, r, np.asarray(edge_list[t][s][r], dtype=np.int64).reshape(-1, 2))
            for t in edge_list for s in edge_list[t] for r in edge_list[t][s]]


class _GraphStub:
    def __init__(self, fx):
        self.edge_list = fx["edge_list"]
        self._t, self._m = list(fx["types"]), [tuple(m) for m in fx["meta_graph"]]
        self.node_feature = {t: [] for t in self._t}

    def get_types(self):
        return self._t

    def get_meta_graph(self):
        return self._m


@pytest.fixture(params=["batched", "slices", "numpy"])
def sampler_impl(request, monkeypatch):
    """The three code paths of sampler.py: whole add_budget batches in native code (default), one native call per
    adjacency slice, pure numpy (library absent).  All must reproduce the reference bit for bit."""
    if request.param != "batched":
        monkeypatch.setattr(sampler, "_NATIVE_BATCH", [None, True])
    if request.param == "numpy":
        monkeypatch.setattr(sampler, "_NATIVE", [None, True])
    if request.param == "batched" and sampler._native_batch() is None:
        pytest.skip("libhgt_b200.so not built")
    return request.param


def test_sampler_reproduces_reference_golden(sampler_impl):
    fx = load_golden("sampler")
    g = _GraphStub(fx)
    fg = sampler.FrozenGraph(g)
    for case in fx["cases"]:
        np.random.seed(case["np_seed"])
        feature, times, edge_list, indxs, texts = sampler.sample_subgraph(fg, fx["time_range"], case["depth"],
                                                                          case["number"], fx["inp"], _extractor)
        assert np.array_equal(np.random.get_state()[1], case["rng_after"]), "RNG stream consumed differently"
        assert list(feature.keys()) == list(case["feature"].keys())
        for k in feature:
            assert np.array_equal(feature[k], case["feature"][k]) and np.array_equal(indxs[k], case["indxs"][k])
            assert np.array_equal(times[k], case["times"][k])
        got, ref = _norm(edge_list), case["edge_list"]
        assert [x[:3] for x in got] == [tuple(x[:3]) for x in ref]
        for a, b in zip(got, ref):
            assert np.array_equal(a[3], b[3]), a[:3]
        # ... and the ingest on top of it gives the reference's tensors
        out = hdata.to_torch(feature, times, edge_list, g)
        assert torch.equal(out[1], case["node_type"]) and torch.equal(out[2], case["edge_time"])
        assert torch.equal(out[3], case["edge_index"]) and torch.equal(out[4], case["edge_type"])


def test_sampler_matches_reference_on_a_larger_graph(sampler_impl):
    """A 10k-node graph sampled 5 deep, 64 per type: the reference's blocks, sampled ids and final RNG state, recorded
    as digests in tests/golden/reference_record.json (oracle/make_golden.py:reference_record)."""
    from oracle import make_golden as mg
    rec = load_record()["sampler_large"]
    edge_list, time_range, inp = mg.sampler_large_inputs()
    fg = sampler.FrozenGraph(types.SimpleNamespace(edge_list=edge_list))
    np.random.seed(rec["np_seed"])
    _, _, s_edges, s_indxs, _ = sampler.sample_subgraph(fg, time_range, rec["depth"], rec["number"], inp, _extractor)
    got = mg.sampler_digests(s_edges, s_indxs, np.random.get_state()[1])
    assert got["rng_after"] == rec["rng_after"], "RNG stream consumed differently"
    assert [b[:3] for b in got["blocks"]] == [b[:3] for b in rec["blocks"]]
    assert got["blocks"] == rec["blocks"]
    assert got["indxs"] == rec["indxs"]


def test_frozen_graph_from_plain_graph_argument():
    """Passing the reference Graph itself (not a FrozenGraph) freezes it on the fly: same result."""
    fx = load_golden("sampler")
    g = _GraphStub(fx)
    case = fx["cases"][0]
    np.random.seed(case["np_seed"])
    out = sampler.sample_subgraph(g, fx["time_range"], case["depth"], case["number"], fx["inp"], _extractor)
    assert all(np.array_equal(out[3][k], case["indxs"][k]) for k in case["indxs"])


def _run_both(g, fx, inp):
    outs = []
    for impl in ("active", "slices"):
        saved = sampler._NATIVE_BATCH[:]
        if impl == "slices":
            sampler._NATIVE_BATCH[:] = [None, True]
        try:
            np.random.seed(21)
            out = sampler.sample_subgraph(sampler.FrozenGraph(g), fx["time_range"], 2, 8, inp, _extractor)
            outs.append((out, np.random.get_state()[1].copy()))
        finally:
            sampler._NATIVE_BATCH[:] = saved
    (a, rng_a), (b, rng_b) = outs
    assert np.array_equal(rng_a, rng_b)
    assert list(a[3].keys()) == list(b[3].keys()) and all(np.array_equal(a[3][k], b[3][k]) for k in a[3])
    na, nb = _norm(a[2]), _norm(b[2])
    assert [x[:3] for x in na] == [x[:3] for x in nb] and all(np.array_equal(x[3], y[3]) for x, y in zip(na, nb))
    return a


def test_seed_ids_beyond_the_graph_and_unknown_seed_types():
    """Seeds the frozen graph has never seen (an id past every adjacency, a type without edges) become isolated sampled
    nodes, as in the reference (`graph.edge_list[_type]` is a defaultdict): the batched native path (which grows its
    state arrays / hands unknown types to the per-slice path) agrees with the per-slice implementation."""
    fx = load_golden("sampler")
    g = _GraphStub(fx)
    first = next(iter(fx["inp"]))
    big = max(sampler.FrozenGraph(g).n_ids.values()) + 7
    seeds = np.concatenate([np.asarray(fx["inp"][first]), [[big, 2010]]])
    a = _run_both(g, fx, {first: seeds})
    assert big in a[3][first].tolist()
    a = _run_both(g, fx, {first: seeds, "never_seen_type": np.array([[3, 2011]])})
    assert big in a[3][first].tolist() and a[3]["never_seen_type"].tolist() == [3]
