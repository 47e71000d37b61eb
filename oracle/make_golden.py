"""Generate tests/golden/*.pt by running the UNMODIFIED reference (/root/reference/pyHGT/conv.py,
model.py) on CPU behind oracle/pyg_shim.py.  TEST INFRASTRUCTURE ONLY.

Run in the dev container (the reference tree does not travel to the GPU box):
    python -m oracle.make_golden

Each fixture holds: cfg (constructor args), state_dict (reference parameter names), the five input
tensors, out [N,d], att [E,H], and — where ``grads`` is set — d(sum(out*w))/d{node_inp, params}.
Sizes are kept to a few hundred KB each so they can be committed.
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import pyg_shim                      # noqa: E402
from pyhgt_b200 import synth                      # noqa: E402

OUT_DIR = os.path.join(ROOT, "tests", "golden")


def _perturb(module, seed):
    """Move skip / relation_pri / LayerNorm affine / biases away from their constant inits so a
    missing term cannot hide behind a 1 or a 0."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in module.named_parameters():
            if name.endswith("skip") or name.endswith("relation_pri") or "norms" in name or "norm." in name:
                p.add_(torch.randn(p.shape, generator=g) * 0.3)


def conv_case(name, graph, d, heads, use_norm, use_RTE, seed, grads=False, feat_scale=1.0):
    conv, _ = pyg_shim.load_reference()
    torch.manual_seed(seed)
    m = conv.HGTConv(d, d, graph.num_types, graph.num_relations, heads, 0.2, use_norm, use_RTE)
    _perturb(m, seed + 1)
    m.eval()
    g = torch.Generator().manual_seed(seed + 2)
    x = torch.randn(graph.num_nodes, d, generator=g) * feat_scale
    fx = {"cfg": dict(in_dim=d, out_dim=d, num_types=graph.num_types, num_relations=graph.num_relations,
                      n_heads=heads, use_norm=use_norm, use_RTE=use_RTE),
          "state_dict": {k: v.detach().clone() for k, v in m.state_dict().items()},
          "node_inp": x, "node_type": graph.node_type, "edge_index": graph.edge_index,
          "edge_type": graph.edge_type, "edge_time": graph.edge_time}
    if grads:
        x = x.clone().requires_grad_(True)
        w = torch.randn(graph.num_nodes, d, generator=g)
        out = m(x, graph.node_type, graph.edge_index, graph.edge_type, graph.edge_time)
        (out * w).sum().backward()
        fx["grad_weight"] = w
        fx["grad_node_inp"] = x.grad.detach().clone()
        fx["grad_params"] = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
        fx["out"] = out.detach().clone()
    else:
        with torch.no_grad():
            fx["out"] = m(x, graph.node_type, graph.edge_index, graph.edge_type, graph.edge_time).clone()
    fx["att"] = m.att.detach().clone()
    path = os.path.join(OUT_DIR, name + ".pt")
    torch.save(fx, path)
    print("%-28s N=%d E=%d d=%d H=%d  %.0f KB" % (name, graph.num_nodes, graph.num_edges, d, heads,
                                                 os.path.getsize(path) / 1024))


def dense_case(name, graph, d, heads, use_norm, use_RTE, seed):
    """DenseHGTConv.forward (conv.py:143-280): same message(), residual + LayerNorm + shared FFN update."""
    conv, _ = pyg_shim.load_reference()
    torch.manual_seed(seed)
    m = conv.DenseHGTConv(d, d, graph.num_types, graph.num_relations, heads, 0.2, use_norm, use_RTE)
    _perturb(m, seed + 1)
    m.eval()
    g = torch.Generator().manual_seed(seed + 2)
    x = torch.randn(graph.num_nodes, d, generator=g)
    with torch.no_grad():
        out = m(x, graph.node_type, graph.edge_index, graph.edge_type, graph.edge_time).clone()
    fx = {"cfg": dict(in_dim=d, out_dim=d, num_types=graph.num_types, num_relations=graph.num_relations,
                      n_heads=heads, use_norm=use_norm, use_RTE=use_RTE),
          "state_dict": {k: v.detach().clone() for k, v in m.state_dict().items()},
          "node_inp": x, "node_type": graph.node_type, "edge_index": graph.edge_index,
          "edge_type": graph.edge_type, "edge_time": graph.edge_time, "out": out, "att": m.att.detach().clone()}
    # gradients of sum(out * w) from the reference's own autograd (training path of the dense variant)
    xg = x.clone().requires_grad_(True)
    w = torch.randn(graph.num_nodes, d, generator=g)
    (m(xg, graph.node_type, graph.edge_index, graph.edge_type, graph.edge_time) * w).sum().backward()
    fx["grad_weight"] = w
    fx["grad_node_inp"] = xg.grad.detach().clone()
    fx["grad_params"] = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
    path = os.path.join(OUT_DIR, name + ".pt")
    torch.save(fx, path)
    print("%-28s N=%d E=%d d=%d H=%d  %.0f KB" % (name, graph.num_nodes, graph.num_edges, d, heads,
                                                 os.path.getsize(path) / 1024))


def gnn_case(name, graph, in_dim, n_hid, heads, n_layers, seed):
    """GNN.forward (model.py:69-80): per-type adapter + stack of GeneralConv('hgt')."""
    _, model = pyg_shim.load_reference()
    torch.manual_seed(seed)
    m = model.GNN(in_dim, n_hid, graph.num_types, graph.num_relations, heads, n_layers, 0.2,
                  "hgt", True, False, True)
    _perturb(m, seed + 1)
    m.eval()
    g = torch.Generator().manual_seed(seed + 2)
    x = torch.randn(graph.num_nodes, in_dim, generator=g)
    with torch.no_grad():
        out = m(x, graph.node_type, graph.edge_time, graph.edge_index, graph.edge_type)
    fx = {"cfg": dict(in_dim=in_dim, n_hid=n_hid, num_types=graph.num_types, num_relations=graph.num_relations,
                      n_heads=heads, n_layers=n_layers, prev_norm=True, last_norm=False, use_RTE=True),
          "state_dict": {k: v.detach().clone() for k, v in m.state_dict().items()},
          "node_feature": x, "node_type": graph.node_type, "edge_index": graph.edge_index,
          "edge_type": graph.edge_type, "edge_time": graph.edge_time, "out": out.clone()}
    xg = x.clone().requires_grad_(True)
    w = torch.randn(graph.num_nodes, n_hid, generator=g)
    (m(xg, graph.node_type, graph.edge_time, graph.edge_index, graph.edge_type) * w).sum().backward()
    fx["grad_weight"] = w
    fx["grad_node_feature"] = xg.grad.detach().clone()
    fx["grad_params"] = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
    path = os.path.join(OUT_DIR, name + ".pt")
    torch.save(fx, path)
    print("%-28s N=%d E=%d  %.0f KB" % (name, graph.num_nodes, graph.num_edges, os.path.getsize(path) / 1024))


def synthetic_sampled_subgraph(seed, n_per_type=(40, 25, 10), n_edges=300):
    """A sampled sub-graph in the format sample_subgraph() returns (data.py:210): feature / times per type and
    edge_list[target_type][source_type][relation] = [[target_ser, source_ser], ...], plus a reference Graph object that
    defines the type order and the meta graph."""
    data = pyg_shim.load_reference_data()
    g = data.Graph()
    names = ["paper", "author", "venue"]
    rels = [("author", "paper", "AP_write"), ("paper", "paper", "PP_cite"), ("paper", "venue", "PV_Journal")]
    for s_t, t_t, r in rels:                                    # defines get_meta_graph() (incl. rev_ relations)
        g.add_edge({"type": s_t, "id": "s0"}, {"type": t_t, "id": "t0"}, time=2000, relation_type=r)
    for t in names:
        g.node_feature[t] = []                                  # get_types() = list(node_feature.keys())
    feature, times, edge_list = sampled_subgraph_inputs(seed, g.get_types(), g.get_meta_graph(), n_per_type, n_edges)
    return data, g, feature, times, edge_list


def sampled_subgraph_inputs(seed, types, metas, n_per_type, n_edges):
    """The seeded part of synthetic_sampled_subgraph: needs only the type order and the meta graph (both stored in
    tests/golden/to_torch.pt), not the reference."""
    import numpy as np
    from collections import defaultdict
    rng = np.random.RandomState(seed)
    feature = {t: rng.randn(n, 7).astype(np.float32) for t, n in zip(types, n_per_type)}
    times = {t: rng.randint(1990, 2020, size=n) for t, n in zip(types, n_per_type)}
    sizes = dict(zip(types, n_per_type))
    edge_list = defaultdict(lambda: defaultdict(lambda: defaultdict(lambda: [])))
    for _ in range(n_edges):
        t_t, s_t, r = metas[rng.randint(len(metas))]
        edge_list[t_t][s_t][r] += [[int(rng.randint(sizes[t_t])), int(rng.randint(sizes[s_t]))]]
    for t in types:                                             # 'self' loops as in data.py:183-186
        for i in range(sizes[t]):
            edge_list[t][t]['self'] += [[i, i]]
    return feature, times, edge_list


def to_torch_case(name, seed):
    data, g, feature, times, edge_list = synthetic_sampled_subgraph(seed)
    ref = data.to_torch(feature, times, edge_list, g)
    plain_edges = {t: {s: {r: [list(map(int, p)) for p in lst] for r, lst in d2.items()} for s, d2 in d1.items()}
                   for t, d1 in edge_list.items()}
    fx = {"feature": feature, "time": times, "edge_list": plain_edges, "types": g.get_types(),
          "meta_graph": g.get_meta_graph(), "node_feature": ref[0], "node_type": ref[1], "edge_time": ref[2],
          "edge_index": ref[3], "edge_type": ref[4], "node_dict": ref[5], "edge_dict": ref[6]}
    path = os.path.join(OUT_DIR, name + ".pt")
    torch.save(fx, path)
    print("%-28s N=%d E=%d  %.0f KB" % (name, ref[1].numel(), ref[4].numel(), os.path.getsize(path) / 1024))


def sampler_graph(data, seed, n_paper=300, n_author=200, n_venue=8, n_field=30, e_ap=1200, e_pp=900, e_pf=700):
    """A small OAG-like reference Graph built through the reference's own add_edge (rev_ relations included)."""
    import numpy as np
    rng = np.random.RandomState(seed)
    g = data.Graph()
    years = rng.randint(2000, 2020, size=n_paper)

    def paper(i):
        return {"type": "paper", "id": "p%d" % i}
    for i in range(n_paper):
        g.add_edge(paper(i), {"type": "venue", "id": "v%d" % rng.randint(n_venue)}, time=int(years[i]),
                   relation_type="PV_Journal")
    for _ in range(e_ap):
        p = rng.randint(n_paper)
        g.add_edge({"type": "author", "id": "a%d" % rng.randint(n_author)}, paper(p), time=int(years[p]),
                   relation_type="AP_write")
    for _ in range(e_pp):
        p, q = rng.randint(n_paper), rng.randint(n_paper)
        g.add_edge(paper(p), paper(q), time=int(years[q]), relation_type="PP_cite")
    for _ in range(e_pf):
        p = rng.randint(n_paper)
        g.add_edge(paper(p), {"type": "field", "id": "f%d" % rng.randint(n_field)},
                   time=None if rng.rand() < 0.3 else int(years[p]), relation_type="PF_in_L2")
    for t in ("paper", "author", "venue", "field"):
        g.node_feature[t] = []
    return g, years


def sampler_extractor(layer_data, graph):
    """Stand-in for feature_OAG (data.py:55-84; needs pandas frames and removed numpy aliases): ids and times as the
    feature, same dict / ordering conventions."""
    import numpy as np
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


def sampler_case(name, seed):
    """sample_subgraph (data.py:87-210) run by the UNMODIFIED reference with a seeded numpy RNG, then the reference's
    to_torch on the result.  The fixture stores the graph's edge_list as plain nested dicts (insertion orders kept)."""
    import numpy as np
    data = pyg_shim.load_reference_data()
    g, years = sampler_graph(data, seed)
    time_range = {int(y): True for y in range(2000, 2016)}
    pids = np.random.RandomState(100 + seed).choice(300, 24, replace=False)
    inp = {"paper": np.array([[int(p), int(years[p])] for p in pids])}
    cases = []
    for depth, number in ((2, 8), (4, 16)):
        np.random.seed(7 + seed)
        feature, times, edge_list, indxs, _ = data.sample_subgraph(g, time_range, depth, number, inp, sampler_extractor)
        rng_after = np.random.get_state()[1].copy()
        tt = data.to_torch(feature, times, edge_list, g)
        cases.append({"depth": depth, "number": number, "np_seed": 7 + seed,
                      "feature": feature, "times": times, "indxs": indxs,
                      "edge_list": [(t, s, r, np.asarray(edge_list[t][s][r], dtype=np.int64).reshape(-1, 2))
                                    for t in edge_list for s in edge_list[t] for r in edge_list[t][s]],
                      "rng_after": rng_after, "node_type": tt[1], "edge_time": tt[2], "edge_index": tt[3],
                      "edge_type": tt[4]})
    plain = {t: {s_: {r: {tid: dict(adl) for tid, adl in tesr.items()} for r, tesr in d2.items()}
                 for s_, d2 in d1.items()} for t, d1 in g.edge_list.items()}
    fx = {"edge_list": plain, "types": g.get_types(), "meta_graph": g.get_meta_graph(), "time_range": time_range,
          "inp": inp, "cases": cases}
    path = os.path.join(OUT_DIR, name + ".pt")
    torch.save(fx, path)
    print("%-28s %d sampled cases  %.0f KB" % (name, len(cases), os.path.getsize(path) / 1024))


def sampler_edge_list(seed, n_paper, n_author, n_venue, n_field, e_ap, e_pp, e_pf):
    """An OAG-like graph straight in the reference's adjacency layout (data.py:35-38), without the reference:
    edge_list[target_type][source_type][relation][target_id][source_id] = time, each edge also stored the other way
    round under 'rev_' + relation.  Node ids are the drawn ids.  Returns (edge_list, paper years)."""
    import numpy as np
    rng = np.random.RandomState(seed)
    years = rng.randint(2000, 2020, size=n_paper)
    edge_list = {}

    def link(s_t, s, t_t, t, time, r):
        for a_t, a, b_t, b, rel in ((t_t, t, s_t, s, r), (s_t, s, t_t, t, "rev_" + r)):
            edge_list.setdefault(a_t, {}).setdefault(b_t, {}).setdefault(rel, {}).setdefault(a, {})[b] = time
    for i in range(n_paper):
        link("paper", i, "venue", int(rng.randint(n_venue)), int(years[i]), "PV_Journal")
    for _ in range(e_ap):
        p = int(rng.randint(n_paper))
        link("author", int(rng.randint(n_author)), "paper", p, int(years[p]), "AP_write")
    for _ in range(e_pp):
        p, q = int(rng.randint(n_paper)), int(rng.randint(n_paper))
        link("paper", p, "paper", q, int(years[q]), "PP_cite")
    for _ in range(e_pf):
        p = int(rng.randint(n_paper))
        link("paper", p, "field", int(rng.randint(n_field)), None if rng.rand() < 0.3 else int(years[p]), "PF_in_L2")
    return edge_list, years


# The larger cases of tests/test_data_ingest.py and tests/test_sampler.py.  Their outputs are too large to store, so
# the record keeps SHA-256 digests of them; the inputs are regenerated from these arguments.
TO_TORCH_LARGE = dict(seed=5, n_per_type=[3000, 2000, 300], n_edges=60000)
SAMPLER_LARGE = dict(graph=dict(seed=11, n_paper=6000, n_author=4000, n_venue=20, n_field=200, e_ap=24000,
                                e_pp=30000, e_pf=18000),
                     seeds=dict(seed=5, count=128), np_seed=3, depth=5, number=64)


def sampler_large_inputs():
    """(edge_list, time_range, inp) of SAMPLER_LARGE."""
    import numpy as np
    edge_list, years = sampler_edge_list(**SAMPLER_LARGE["graph"])
    time_range = {int(y): True for y in range(2000, 2016)}
    pids = np.random.RandomState(SAMPLER_LARGE["seeds"]["seed"]).choice(SAMPLER_LARGE["graph"]["n_paper"],
                                                                       SAMPLER_LARGE["seeds"]["count"], replace=False)
    inp = {"paper": np.array([[int(p), int(years[p])] for p in pids])}
    return edge_list, time_range, inp


def digest(a):
    """SHA-256 over an array's dtype, shape and bytes (numpy array or CPU tensor)."""
    import hashlib
    import numpy as np
    a = np.ascontiguousarray(a.numpy() if isinstance(a, torch.Tensor) else a)
    h = hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def sampler_digests(edge_list, indxs, rng_state):
    """What tests/test_sampler.py compares of one sample_subgraph result: the sampled blocks in order, the sampled ids
    per type and numpy's RNG state afterwards."""
    import numpy as np
    blocks = [[t, s, r, digest(np.asarray(edge_list[t][s][r], dtype=np.int64).reshape(-1, 2))]
              for t in edge_list for s in edge_list[t] for r in edge_list[t][s]]
    return {"blocks": blocks, "indxs": {k: digest(np.asarray(v, dtype=np.int64)) for k, v in indxs.items()},
            "rng_after": digest(np.asarray(rng_state, dtype=np.uint32))}


def _inventory(module):
    return [[n, list(p.shape)] for n, p in module.named_parameters()]


def reference_record(name):
    """Facts about the reference that tests check without it: parameter inventories (names and shapes) and digests of
    the reference's outputs on TO_TORCH_LARGE and SAMPLER_LARGE."""
    import json
    import types
    import warnings
    import numpy as np
    conv, model = pyg_shim.load_reference()
    data = pyg_shim.load_reference_data()
    rec = {"hgtconv_32_3_4_4_params": _inventory(conv.HGTConv(32, 32, 3, 4, 4, 0.2, True, True)),
           "mag_gnn_params": _inventory(model.GNN(in_dim=129, n_hid=512, num_types=4, num_relations=9, n_heads=8,
                                                  n_layers=4, prev_norm=True, last_norm=True, use_RTE=True)),
           "mag_classifier_params": _inventory(model.Classifier(512, 349))}

    _, g, feature, times, edge_list = synthetic_sampled_subgraph(**TO_TORCH_LARGE)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = data.to_torch(feature, times, edge_list, g)
    keys = ("node_feature", "node_type", "edge_time", "edge_index", "edge_type")
    rec["to_torch_large"] = dict(TO_TORCH_LARGE, **{k: digest(v) for k, v in zip(keys, ref[:5])},
                                 node_dict={k: [int(x) for x in v] for k, v in ref[5].items()},
                                 edge_dict={k: int(v) for k, v in ref[6].items()})

    edge_list, time_range, inp = sampler_large_inputs()
    np.random.seed(SAMPLER_LARGE["np_seed"])
    _, _, s_edges, s_indxs, _ = data.sample_subgraph(types.SimpleNamespace(edge_list=edge_list), time_range,
                                                     SAMPLER_LARGE["depth"], SAMPLER_LARGE["number"], inp,
                                                     sampler_extractor)
    rec["sampler_large"] = dict(SAMPLER_LARGE, **sampler_digests(s_edges, s_indxs, np.random.get_state()[1]))
    path = os.path.join(OUT_DIR, name + ".json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")
    print("%-28s %.0f KB" % (name, os.path.getsize(path) / 1024))


def main():
    os.makedirs(OUT_DIR, exist_ok=True)
    to_torch_case("to_torch", seed=31)
    sampler_case("sampler", seed=3)
    c1 = synth.make_c1()
    conv_case("c1_norte", c1, 64, 4, True, False, seed=10)              # BASELINE config 1
    conv_case("c1_rte", c1, 64, 4, True, True, seed=11, grads=True)
    # unsorted types, all <s,t,r> triples, isolated destinations, self loops, multi-edges, d_k=4
    g = synth.make_random(300, 2500, 3, 4, seed=21, isolated_frac=0.3, self_loops=40, duplicate_edges=60)
    conv_case("rand_t3r4_dk4", g, 32, 8, False, True, seed=12, grads=True)
    # odd head width (d_k = 25 -> scalar lanes) and larger feature magnitude
    g = synth.make_random(200, 1500, 2, 3, seed=22, sorted_types=True)
    conv_case("rand_dk25", g, 100, 4, True, False, seed=13, feat_scale=2.0)
    # OAG head width d_k = 50 (d=100, H=2) with RTE, mag-shaped miniature (authors have no in-edges)
    g = synth.make_mag_shaped(scale=2e-4, seed=23)
    conv_case("mag_mini_dk50", g, 100, 2, True, True, seed=14)
    # oag-shaped miniature, d_k = 16, 6 types / 10 relations incl. self relation
    g = synth.make_oag_shaped(scale=2e-3, seed=24)
    conv_case("oag_mini", g, 64, 4, True, True, seed=15)
    # a hub: one destination receives 3000 of the edges (segment splitting), H=2
    g = synth.make_random(400, 1000, 2, 2, seed=25)
    hub = torch.full((3000,), 7, dtype=torch.int64)
    gen = torch.Generator().manual_seed(99)
    g.edge_index = torch.cat([g.edge_index, torch.stack([torch.randint(0, 400, (3000,), generator=gen), hub])], 1)
    g.edge_type = torch.cat([g.edge_type, torch.randint(0, 2, (3000,), generator=gen)])
    g.edge_time = torch.cat([g.edge_time, torch.randint(0, 240, (3000,), generator=gen)])
    conv_case("hub_h2", g, 64, 2, True, True, seed=16)
    # whole-model fixture: reference GNN (adapter + 2 HGT layers)
    g = synth.make_random(250, 2000, 3, 3, seed=26, sorted_types=True, self_loops=250)
    gnn_case("gnn_2layer", g, 48, 64, 4, 2, seed=17)
    # DenseHGTConv variant (unsorted types, isolated destinations), d=64 so the FFN runs on the tensor-core GEMM
    g = synth.make_random(300, 2400, 3, 3, seed=27, isolated_frac=0.2, self_loops=30)
    dense_case("dense_hgt", g, 64, 4, True, True, seed=18)
    reference_record("reference_record")


if __name__ == "__main__":
    main()
