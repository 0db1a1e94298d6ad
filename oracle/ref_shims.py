"""TEST INFRASTRUCTURE ONLY - never imported by the product package.

Loader for the *unmodified* reference modules (`/root/reference/gcn_lib`) in a
container that lacks the reference's third-party CUDA extensions.  It injects
small stand-ins for the absent packages into ``sys.modules`` and then imports
the reference's own ``gcn_lib.dense`` / ``gcn_lib.sparse`` so that the
reference code itself executes on CPU torch.  Used by

* ``tests/golden/gen_golden.py`` and ``tests/golden/gen_golden_models.py`` -
  to generate the committed golden vectors and API fixture that the tests
  compare against; no test loads the reference itself.

Third-party arithmetic restated here (none of it lives under /root/reference;
versions are NOT pinned by the reference: deepgcn_env_install.sh:21-32 installs
"latest" torch-scatter / torch-geometric for torch-1.9.0+cu102):

* ``torch_scatter.scatter(src, index, dim, dim_size, reduce)``
  sum / mean (count clamped to >=1) / max / min, empty groups -> 0.
  call sites: gcn_lib/sparse/torch_message.py:57,71
* ``torch_scatter.scatter_softmax(src, index, dim)``
  exp(src - groupmax) / groupsum(exp(src - groupmax)).
  call sites: gcn_lib/sparse/torch_message.py:52,55
* ``torch_geometric.utils.degree(index, num_nodes)`` - float in-degree count.
  call sites: gcn_lib/sparse/torch_message.py:62,79
* ``torch_geometric.nn.MessagePassing.propagate`` (flow source_to_target):
  x_j = x.index_select(0, edge_index[0]); message(); aggregate(index =
  edge_index[1], dim_size = N); update().
  call site: gcn_lib/sparse/torch_vertex.py:68
* ``torch_cluster.knn_graph(x, k, loop=False, flow='source_to_target')``:
  row 0 = neighbour, row 1 = centre, grouped by centre, self excluded.
  call sites: gcn_lib/dense/torch_edge.py:90,97
"""
import importlib
import os
import sys
import types

import torch

REFERENCE_ROOT = os.environ.get("DGCN_REFERENCE_ROOT", "/root/reference")


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "gcn_lib"))


# --------------------------------------------------------------------------
# torch_scatter stand-in
# --------------------------------------------------------------------------
def _expand_index(index, src, dim):
    if index.dim() == src.dim():
        return index
    shape = [1] * src.dim()
    shape[dim] = -1
    return index.view(shape).expand_as(src)


def scatter(src, index, dim=-1, out=None, dim_size=None, reduce="sum"):
    dim = dim % src.dim()
    if dim_size is None:
        dim_size = int(index.max()) + 1 if index.numel() > 0 else 0
    idx = _expand_index(index, src, dim)
    shape = list(src.shape)
    shape[dim] = dim_size
    if reduce in ("sum", "add"):
        return torch.zeros(shape, dtype=src.dtype).scatter_add_(dim, idx, src)
    if reduce == "mean":
        s = torch.zeros(shape, dtype=src.dtype).scatter_add_(dim, idx, src)
        cnt = torch.zeros(dim_size, dtype=src.dtype).scatter_add_(
            0, index, torch.ones_like(index, dtype=src.dtype)).clamp_(min=1)
        cshape = [1] * src.dim()
        cshape[dim] = -1
        return s / cnt.view(cshape)
    if reduce in ("max", "min"):
        red = "amax" if reduce == "max" else "amin"
        o = torch.zeros(shape, dtype=src.dtype)
        return o.scatter_reduce_(dim, idx, src, reduce=red, include_self=False)
    raise ValueError(reduce)


def scatter_add(src, index, dim=-1, out=None, dim_size=None):
    return scatter(src, index, dim, out, dim_size, "sum")


def scatter_mean(src, index, dim=-1, out=None, dim_size=None):
    return scatter(src, index, dim, out, dim_size, "mean")


def scatter_max(src, index, dim=-1, out=None, dim_size=None):
    return scatter(src, index, dim, out, dim_size, "max"), None


def scatter_min(src, index, dim=-1, out=None, dim_size=None):
    return scatter(src, index, dim, out, dim_size, "min"), None


def scatter_softmax(src, index, dim=-1, eps=0.0):
    dim = dim % src.dim()
    idx = _expand_index(index, src, dim)
    n = int(index.max()) + 1 if index.numel() > 0 else 0
    shape = list(src.shape)
    shape[dim] = n
    gmax = torch.full(shape, float("-inf"), dtype=src.dtype).scatter_reduce_(
        dim, idx, src, reduce="amax", include_self=True)
    rec = (src - gmax.gather(dim, idx)).exp()
    gsum = torch.zeros(shape, dtype=src.dtype).scatter_add_(dim, idx, rec)
    return rec / (gsum.gather(dim, idx) + eps)


# --------------------------------------------------------------------------
# torch_geometric stand-in
# --------------------------------------------------------------------------
class MessagePassing(torch.nn.Module):
    def __init__(self, aggr="add", flow="source_to_target", node_dim=0, **kw):
        super().__init__()
        self.aggr = aggr
        self.flow = flow
        self.node_dim = node_dim

    def propagate(self, edge_index, size=None, **kwargs):
        x = kwargs.get("x")
        n = x.size(self.node_dim) if size is None else size[1]
        msg_kwargs = {}
        if x is not None:
            msg_kwargs["x_j"] = x.index_select(self.node_dim, edge_index[0])
            msg_kwargs["x_i"] = x.index_select(self.node_dim, edge_index[1])
        for key, val in kwargs.items():
            if key != "x":
                msg_kwargs[key] = val
        import inspect
        want = inspect.signature(self.message).parameters
        out = self.message(**{a: v for a, v in msg_kwargs.items() if a in want})
        out = self.aggregate(out, edge_index[1], dim_size=n)
        return self.update(out)

    def message(self, x_j):
        return x_j

    def aggregate(self, inputs, index, ptr=None, dim_size=None):
        red = {"add": "sum", None: "sum"}.get(self.aggr, self.aggr)
        return scatter(inputs, index, dim=self.node_dim, dim_size=dim_size, reduce=red)

    def update(self, inputs):
        return inputs


def degree(index, num_nodes=None, dtype=None):
    n = int(index.max()) + 1 if num_nodes is None else num_nodes
    out = torch.zeros(n, dtype=dtype or torch.get_default_dtype())
    return out.scatter_add_(0, index, torch.ones(index.numel(), dtype=out.dtype))


def remove_self_loops(edge_index, edge_attr=None):
    mask = edge_index[0] != edge_index[1]
    return edge_index[:, mask], (None if edge_attr is None else edge_attr[mask])


def add_self_loops(edge_index, edge_attr=None, fill_value=None, num_nodes=None):
    n = int(edge_index.max()) + 1 if num_nodes is None else num_nodes
    loop = torch.arange(n, dtype=edge_index.dtype).unsqueeze(0).repeat(2, 1)
    return torch.cat([edge_index, loop], dim=1), edge_attr


def knn_graph(x, k, batch=None, loop=False, flow="source_to_target", **kw):
    """k nearest by squared L2 distance (fp64), self excluded unless loop."""
    xd = x.double()
    d = torch.cdist(xd, xd).pow_(2)
    if not loop:
        d.fill_diagonal_(float("inf"))
    nn_idx = d.topk(k, dim=1, largest=False).indices
    centre = torch.arange(x.size(0)).view(-1, 1).expand(-1, k)
    return torch.stack((nn_idx.reshape(-1), centre.reshape(-1)), 0)


class _Placeholder(torch.nn.Module):
    def __init__(self, *a, **k):
        super().__init__()


def _install_stubs():
    if "torch_scatter" not in sys.modules:
        m = types.ModuleType("torch_scatter")
        for f in (scatter, scatter_add, scatter_mean, scatter_max, scatter_min, scatter_softmax):
            setattr(m, f.__name__, f)
        sys.modules["torch_scatter"] = m
    if "torch_cluster" not in sys.modules:
        m = types.ModuleType("torch_cluster")
        m.knn_graph = knn_graph
        sys.modules["torch_cluster"] = m
    if "torch_geometric" not in sys.modules:
        tg = types.ModuleType("torch_geometric")
        nn = types.ModuleType("torch_geometric.nn")
        nn.MessagePassing = MessagePassing
        for name in ("EdgeConv", "GATConv", "SAGEConv", "GCNConv", "GINConv", "DataParallel"):
            setattr(nn, name, type(name, (_Placeholder,), {}))
        utils = types.ModuleType("torch_geometric.utils")
        utils.degree = degree
        utils.remove_self_loops = remove_self_loops
        utils.add_self_loops = add_self_loops
        data = types.ModuleType("torch_geometric.data")
        for name in ("InMemoryDataset", "Data"):
            setattr(data, name, type(name, (), {}))
        data.extract_zip = lambda *a, **k: None
        tg.nn, tg.utils, tg.data = nn, utils, data
        sys.modules.update({"torch_geometric": tg, "torch_geometric.nn": nn,
                            "torch_geometric.utils": utils, "torch_geometric.data": data})
    if "h5py" not in sys.modules:
        sys.modules["h5py"] = types.ModuleType("h5py")


_loaded = {}


def load_reference():
    """Returns (gcn_lib.dense, gcn_lib.sparse) imported from REFERENCE_ROOT."""
    if "mods" in _loaded:
        return _loaded["mods"]
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    _install_stubs()
    # the reference imports itself as top-level `gcn_lib` / `utils`
    for name in list(sys.modules):
        if name == "gcn_lib" or name.startswith("gcn_lib.") or name == "utils" or name.startswith("utils."):
            if not getattr(sys.modules[name], "__file__", "").startswith(REFERENCE_ROOT):
                del sys.modules[name]
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        dense = importlib.import_module("gcn_lib.dense")
        sparse = importlib.import_module("gcn_lib.sparse")
    finally:
        sys.path.remove(REFERENCE_ROOT)
    _loaded["mods"] = (dense, sparse)
    return dense, sparse
