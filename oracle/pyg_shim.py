"""Stand-ins for the three PyTorch-Geometric primitives pyHGT's conv.py imports,
plus a loader that imports the UNMODIFIED reference modules from /root/reference.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Used solely by ``oracle/make_golden.py``
to generate the fixtures under tests/golden, which needs a checkout of the reference
(PYHGT_REFERENCE_ROOT); the tests themselves read only the fixtures.

Third-party arithmetic restated here (not vendored under /root/reference):
torch-geometric==1.3.2 / torch-scatter==1.3.2 (requirements.txt:5,9).  Call sites in
the reference: conv.py:6,13,57 (MessagePassing/propagate), conv.py:8,108 (softmax),
conv.py:7,53-54 (glorot).

  propagate (flow source_to_target, node_dim=0, aggr='add'):
      X_i -> kwargs['X'].index_select(0, edge_index[1]),  X_j -> index_select(0, edge_index[0]),
      edge_index_i -> edge_index[1]; out = zeros[N].index_add_(0, edge_index[1], message(...));
      return update(out, <update args by name>)
  softmax(src, index): m = scatter_max(src, index)[index]; o = exp(src - m);
      o / (scatter_add(o, index)[index] + 1e-16)
  glorot(t): a = sqrt(6 / (t.size(-2) + t.size(-1))); t.uniform_(-a, a)
"""
import importlib
import inspect
import math
import os
import sys
import types

import torch
import torch.nn as nn

REFERENCE_ROOT = os.environ.get("PYHGT_REFERENCE_ROOT", "/root/reference")


def segment_softmax(src, index, num_nodes=None):
    """torch_geometric.utils.softmax (1.3.x) semantics; used at conv.py:108."""
    n = int(index.max()) + 1 if num_nodes is None else num_nodes
    tail = src.shape[1:]
    idx = index.view(-1, *([1] * len(tail))).expand_as(src)
    mx = torch.full((n, *tail), float("-inf"), dtype=src.dtype, device=src.device)
    mx = mx.scatter_reduce(0, idx, src, reduce="amax", include_self=True)
    out = (src - mx.index_select(0, index)).exp()
    den = torch.zeros((n, *tail), dtype=src.dtype, device=src.device).index_add_(0, index, out)
    return out / (den.index_select(0, index) + 1e-16)


def glorot_(tensor):
    """torch_geometric.nn.inits.glorot; used at conv.py:53-54."""
    if tensor is not None:
        a = math.sqrt(6.0 / (tensor.size(-2) + tensor.size(-1)))
        tensor.data.uniform_(-a, a)


def uniform_(size, tensor):
    if tensor is not None:
        bound = 1.0 / math.sqrt(size)
        tensor.data.uniform_(-bound, bound)


class MessagePassingStandIn(nn.Module):
    """Minimal torch_geometric.nn.conv.MessagePassing: gather by suffix, add-aggregate, update."""

    def __init__(self, aggr="add", flow="source_to_target", node_dim=0, **kwargs):
        super().__init__()
        assert aggr == "add" and flow == "source_to_target" and node_dim == 0
        self._msg_args = list(inspect.signature(self.message).parameters)
        self._upd_args = list(inspect.signature(self.update).parameters)[1:]

    def propagate(self, edge_index, size=None, **kwargs):
        n = None
        feed = {}
        for name in self._msg_args:
            if name == "edge_index_i":
                feed[name] = edge_index[1]
            elif name == "edge_index_j":
                feed[name] = edge_index[0]
            elif name.endswith("_i") or name.endswith("_j"):
                base = kwargs[name[:-2]]
                n = base.size(0) if n is None else n
                feed[name] = base.index_select(0, edge_index[1 if name.endswith("_i") else 0])
            else:
                feed[name] = kwargs[name]
        msg = self.message(**feed)
        out = torch.zeros((n,) + tuple(msg.shape[1:]), dtype=msg.dtype, device=msg.device)
        out.index_add_(0, edge_index[1], msg)
        return self.update(out, **{k: kwargs[k] for k in self._upd_args})


class _InertConv(nn.Module):
    def __init__(self, *a, **k):
        super().__init__()


def install():
    """Register the stand-in modules under the names conv.py:5-8 imports."""
    if "torch_geometric" in sys.modules and not getattr(sys.modules["torch_geometric"], "_hgt_shim", False):
        return  # a real PyG is installed: use it
    tg = types.ModuleType("torch_geometric"); tg._hgt_shim = True
    tg_nn = types.ModuleType("torch_geometric.nn")
    tg_conv = types.ModuleType("torch_geometric.nn.conv")
    tg_inits = types.ModuleType("torch_geometric.nn.inits")
    tg_utils = types.ModuleType("torch_geometric.utils")
    tg_nn.GCNConv = _InertConv
    tg_nn.GATConv = _InertConv
    tg_nn.MessagePassing = MessagePassingStandIn
    tg_conv.MessagePassing = MessagePassingStandIn
    tg_inits.glorot = glorot_
    tg_inits.uniform = uniform_
    tg_utils.softmax = segment_softmax
    tg.nn, tg.utils = tg_nn, tg_utils
    tg_nn.conv, tg_nn.inits = tg_conv, tg_inits
    for m in (tg, tg_nn, tg_conv, tg_inits, tg_utils):
        sys.modules[m.__name__] = m


def reference_available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "pyHGT", "conv.py"))


def load_reference_data():
    """Import /root/reference/pyHGT/data.py unchanged (plotting / table packages it imports at module level but never
    uses on the to_torch path are replaced by empty stand-ins)."""
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    install()
    for name in ("seaborn", "matplotlib", "matplotlib.pyplot", "matplotlib.cm", "texttable", "dill"):
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                m = types.ModuleType(name)
                if name == "texttable":
                    m.Texttable = object
                sys.modules[name] = m
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    return importlib.import_module("pyHGT.data")


def load_reference():
    """Import /root/reference/pyHGT/{conv,model}.py unchanged; returns (conv_module, model_module)."""
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    install()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    conv = importlib.import_module("pyHGT.conv")
    model = importlib.import_module("pyHGT.model")
    return conv, model
