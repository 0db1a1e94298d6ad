"""TEST INFRASTRUCTURE ONLY (parity oracle) - the product package must never
import this module; only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may.

CPU restatement (torch CPU tensors, fp32 by default, fp64 on request) of the
dense message-passing hot path of lightaime/deep_gcns_torch.  Every function
names the reference lines it follows.  The fp32 flavour issues the same ATen
CPU ops in the same order as the reference so that it is bit-identical to the
reference on the same host; the fp64 flavour adjudicates fp32 near-ties.

Pinned by tests/test_oracle_pins.py against the golden vectors under
tests/golden/ that tests/golden/gen_golden.py produced by running the
UNMODIFIED reference modules (oracle/ref_shims.py).
"""
import torch
import torch.nn.functional as F


# -- graph construction -----------------------------------------------------
def pairwise_distance(x):
    """gcn_lib/dense/torch_edge.py:32-42.  x (B,N,C) -> (B,N,N).
    D = (|x_i|^2 + (-2 x_i.x_j)) + |x_j|^2, in that association order."""
    x_inner = -2 * torch.matmul(x, x.transpose(2, 1))
    x_square = torch.sum(torch.mul(x, x), dim=-1, keepdim=True)
    return x_square + x_inner + x_square.transpose(2, 1)


def knn_matrix(x, K, dtype=None):
    """gcn_lib/dense/torch_edge.py:45-58.  x (B,C,N,1) -> int64 (2,B,N,K):
    plane 0 = K nearest (self included, ascending distance), plane 1 = centre."""
    with torch.no_grad():
        xt = x.transpose(2, 1).squeeze(-1)
        if dtype is not None:
            xt = xt.to(dtype)
        B, N, _ = xt.shape
        _, nn_idx = torch.topk(-pairwise_distance(xt.detach()), k=K)
        center = torch.arange(0, N, device=xt.device).expand(B, K, -1).transpose(2, 1)
    return torch.stack((nn_idx, center), dim=0)


def knn_exclude_self(x, K):
    """gcn_lib/dense/torch_edge.py:79-101 (`DilatedKnnGraph`): per cloud
    torch_cluster.knn_graph(x[i]^T, K) with loop=False, i.e. the K nearest
    points other than the point itself, ascending, row 0 = neighbour, row 1 =
    centre, reshaped (2,N,K) and stacked over the batch -> (2,B,N,K).
    torch_cluster is third-party and absent; distances here are exact fp64
    |x_i - x_j|^2 (torch_cluster's CPU path is a kd-tree on the same metric)."""
    with torch.no_grad():
        xt = x.squeeze(-1).transpose(2, 1).double()
        B, N, _ = xt.shape
        d = (xt.unsqueeze(2) - xt.unsqueeze(1)).pow(2).sum(-1)
        d.diagonal(dim1=1, dim2=2).fill_(float("inf"))
        nn_idx = d.topk(K, dim=-1, largest=False).indices
        center = torch.arange(0, N, device=xt.device).view(1, N, 1).expand(B, N, K)
    return torch.stack((nn_idx, center), dim=0)


def dilation_columns(k, dilation, stochastic=False, epsilon=0.0, training=False):
    """gcn_lib/dense/torch_edge.py:19-29, host side.  Returns the list of
    columns of the sorted K=k*dilation neighbour list that survive.  Consumes
    the CPU generator exactly like the reference: `torch.rand(1)` on EVERY call
    when `stochastic` (it is the left operand of `and`, :21), `randperm(K)` only
    when that draw < epsilon and training."""
    K = k * dilation
    if stochastic:
        if torch.rand(1) < epsilon and training:
            return torch.randperm(K)[:k]
    return torch.arange(0, K, dilation)


def dilated_knn_graph(x, k, dilation=1, stochastic=False, epsilon=0.0, training=False, dtype=None):
    """gcn_lib/dense/torch_edge.py:61-76 (`DenseDilatedKnnGraph.forward`)."""
    edge_index = knn_matrix(x, k * dilation, dtype)
    cols = dilation_columns(k, dilation, stochastic, epsilon, training)
    return edge_index[:, :, :, cols]


# -- vertex ops -------------------------------------------------------------
def batched_index_select(x, idx):
    """gcn_lib/dense/torch_nn.py:75-96.  x (B,C,N,1), idx (B,N,k) -> (B,C,N,k)."""
    B, C, N = x.shape[:3]
    k = idx.shape[-1]
    flat = (idx + torch.arange(0, B, device=idx.device).view(-1, 1, 1) * N).contiguous().view(-1)
    rows = x.transpose(2, 1).contiguous().view(B * N, -1)[flat, :]
    return rows.view(B, N, k, C).permute(0, 3, 1, 2).contiguous()


def activation(z, act, slope=None):
    """gcn_lib/dense/torch_nn.py:9-21: relu | leakyrelu(0.2) | prelu(1 param) | none."""
    if act is None or str(act).lower() == "none":
        return z
    act = act.lower()
    if act == "relu":
        return F.relu(z)
    if act == "leakyrelu":
        return F.leaky_relu(z, 0.2)
    if act == "prelu":
        return F.prelu(z, slope)
    raise NotImplementedError("activation layer [%s] is not found" % act)


def normalization(a, norm, p, training=False):
    """gcn_lib/dense/torch_nn.py:24-33: BatchNorm2d(affine) | InstanceNorm2d(no
    affine).  `p` holds weight/bias/running_mean/running_var (batch only).
    Training-mode batch norm returns batch statistics alongside so callers can
    check running-stat updates."""
    if norm is None or str(norm).lower() == "none":
        return a
    norm = norm.lower()
    if norm == "batch":
        if training:
            return F.batch_norm(a, None, None, p["weight"], p["bias"], True, 0.1, 1e-5)
        return F.batch_norm(a, p["running_mean"], p["running_var"], p["weight"], p["bias"],
                            False, 0.1, 1e-5)
    if norm == "instance":
        return F.instance_norm(a, eps=1e-5)
    raise NotImplementedError("normalization layer [%s] is not found" % norm)


def basic_conv(feat, p, act="relu", norm=None, training=False):
    """gcn_lib/dense/torch_nn.py:48-58: Conv2d(1x1) -> act -> norm."""
    z = F.conv2d(feat, p["weight"], p.get("bias"))
    return normalization(activation(z, act, p.get("slope")), norm, p.get("norm", {}), training)


def edge_conv(x, edge_index, p, act="relu", norm=None, training=False):
    """gcn_lib/dense/torch_vertex.py:31-35."""
    x_i = batched_index_select(x, edge_index[1])
    x_j = batched_index_select(x, edge_index[0])
    y = basic_conv(torch.cat([x_i, x_j - x_i], dim=1), p, act, norm, training)
    return torch.max(y, -1, keepdim=True)[0]


def mr_conv(x, edge_index, p, act="relu", norm=None, training=False):
    """gcn_lib/dense/torch_vertex.py:16-20."""
    x_i = batched_index_select(x, edge_index[1])
    x_j = batched_index_select(x, edge_index[0])
    r = torch.max(x_j - x_i, -1, keepdim=True)[0]
    return basic_conv(torch.cat([x, r], dim=1), p, act, norm, training)


def graph_conv(x, edge_index, p, conv="edge", act="relu", norm=None, training=False):
    """gcn_lib/dense/torch_vertex.py:38-52."""
    if conv == "edge":
        return edge_conv(x, edge_index, p, act, norm, training)
    if conv == "mr":
        return mr_conv(x, edge_index, p, act, norm, training)
    raise NotImplementedError("conv:{} is not supported".format(conv))


def dyn_conv(x, p, k, dilation=1, conv="edge", act="relu", norm=None, training=False,
             stochastic=False, epsilon=0.0, edge_index=None):
    """gcn_lib/dense/torch_vertex.py:55-72 (`DynConv2d.forward`, knn='matrix')."""
    if edge_index is None:
        edge_index = dilated_knn_graph(x, k, dilation, stochastic, epsilon, training)
    return graph_conv(x, edge_index, p, conv, act, norm, training)


def params_from_module(gconv_nn, dtype=None):
    """Pull the functional parameter dict out of a (reference or drop-in)
    `BasicConv` Sequential: nn.0 = Conv2d, then optional act / norm modules
    (gcn_lib/dense/torch_nn.py:50-58; state_dict keys nn.0.*, nn.2.*)."""
    cast = (lambda t: t.detach().to(dtype)) if dtype is not None else (lambda t: t.detach())
    p = {"weight": cast(gconv_nn[0].weight)}
    if gconv_nn[0].bias is not None:
        p["bias"] = cast(gconv_nn[0].bias)
    for m in list(gconv_nn)[1:]:
        if isinstance(m, torch.nn.PReLU):
            p["slope"] = cast(m.weight)
        if isinstance(m, torch.nn.BatchNorm2d):
            p["norm"] = {k: cast(getattr(m, k)) for k in ("weight", "bias", "running_mean", "running_var")}
    return p


# -- comparators used by the parity tests ------------------------------------
def knn_mismatch_report(x, nn_mine, nn_ref, rel_tol=1e-5):
    """Index-parity adjudication (SURVEY.md 7 'kNN index parity').
    x (B,C,N,1) fp32; nn_* int64 (B,N,K) sorted neighbour lists.  Returns
    (n_mismatch, n_unexplained): a mismatching slot is explained when the fp64
    distances of the two candidates at that slot differ by less than
    rel_tol * max(1, |d|) - an fp32 near-tie that no two fp32 evaluation orders
    are obliged to rank identically."""
    xt = x.squeeze(-1).transpose(2, 1).double()
    sq = (xt * xt).sum(-1)
    bad = nn_mine != nn_ref
    n_bad = int(bad.sum())
    if n_bad == 0:
        return 0, 0
    b, i, l = bad.nonzero(as_tuple=True)
    jm, jr = nn_mine[b, i, l], nn_ref[b, i, l]
    def dist(j):
        return sq[b, i] - 2 * (xt[b, i] * xt[b, j]).sum(-1) + sq[b, j]
    dm, dr = dist(jm), dist(jr)
    scale = torch.maximum(torch.ones_like(dm), torch.maximum(dm.abs(), dr.abs()))
    unexplained = ((dm - dr).abs() > rel_tol * scale)
    return n_bad, int(unexplained.sum())
