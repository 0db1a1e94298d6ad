"""Model-level golden vectors: the reference's OWN model assemblies (examples/sem_seg_dense/architecture.py,
examples/modelnet_cls/architecture.py, examples/ogb/ogbn_arxiv/model.py) and its reversible coupling
(eff_gcn_modules/rev/memgcn.py), executed unmodified on the unmodified gcn_lib (loaded through
oracle/ref_shims.py), on seeded synthetic inputs.  Small configurations of BASELINE configs 2, 3, 4:

    model_resgcn4     DenseDeepGCN: 4 blocks (head + 3 ResDynBlock2d, dilation 1..3), edge conv, k=8, 32 filters
    model_mrgcn4      DeepGCN (modelnet_cls): DilatedKnnGraph head (self excluded) + 3 ResDynBlock2d('mr'), k=6
    model_deepergcn8  DeeperGCN 'res+': 8 GENConv(softmax_sg, t=0.1, mlp_layers=1) + BatchNorm1d
    model_revgnn      GroupAdditiveCoupling(group=2) over two GENConv(C/2): forward and inverse

    python tests/golden/gen_golden_models.py        # needs /root/reference

Each file: `in.*`, `sd.*` (the reference model's state_dict: the drop-in model must load it with strict=True),
`out.*`, `meta`.
"""
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)
from oracle import ref_shims  # noqa: E402
from gen_golden import randomize_norm, save  # noqa: E402


def load_source(rel, drop_main=True):
    src = open(os.path.join(ref_shims.REFERENCE_ROOT, rel)).read()
    if drop_main:
        src = src.split("if __name__ ==")[0]
    return src.replace("import __init__\n", "")


def exec_reference(rel, name):
    ns = {"__name__": name}
    sys.path.insert(0, ref_shims.REFERENCE_ROOT)
    try:
        exec(compile(load_source(rel), rel, "exec"), ns)
    finally:
        sys.path.remove(ref_shims.REFERENCE_ROOT)
    return ns


def capture(model):
    """Forward hooks on the head / backbone blocks (features) and on every graph builder (neighbour lists)."""
    feats, graphs, handles = [], [], []
    handles.append(model.head.register_forward_hook(lambda m, i, o: feats.append(o.detach().clone())))
    handles.append(model.knn.register_forward_hook(lambda m, i, o: graphs.append(o[0].to(torch.int32).clone())))
    for blk in model.backbone:
        handles.append(blk.register_forward_hook(lambda m, i, o: feats.append(o.detach().clone())))
        handles.append(blk.body.dilated_knn_graph.register_forward_hook(
            lambda m, i, o: graphs.append(o[0].to(torch.int32).clone())))
    return feats, graphs, handles


def main():
    torch.set_num_threads(8)
    ref_shims.load_reference()
    gen = torch.Generator().manual_seed(7)

    # ---- config 2 in small: examples/sem_seg_dense/architecture.py:7-56 --------------------------------------
    ns = exec_reference("examples/sem_seg_dense/architecture.py", "ref_semseg")
    opt = dict(n_filters=32, k=8, act="relu", norm="batch", bias=True, epsilon=0.2, stochastic=True, conv="edge",
               n_blocks=4, block="res", in_channels=9, n_classes=13, dropout=0.3)
    torch.manual_seed(0)
    model = ns["DenseDeepGCN"](types.SimpleNamespace(**opt)).eval()
    randomize_norm(model, gen)
    pos, feat = torch.rand(2, 256, 3, generator=gen), torch.rand(2, 256, 6, generator=gen)
    inputs = torch.cat((pos, feat), 2).transpose(1, 2).unsqueeze(-1).contiguous()
    feats, graphs, handles = capture(model)
    with torch.no_grad():
        torch.manual_seed(5)                      # stochastic dilation draws torch.rand(1) per layer even in eval
        y = model(inputs)
    for h in handles:
        h.remove()
    outs = {"y": y}
    for i, (f, gph) in enumerate(zip(feats, graphs)):
        outs["feat%d" % i], outs["graph%d" % i] = f, gph
    save("model_resgcn4", dict(opt, B=2, N=256), {"inputs": inputs}, model.state_dict(), outs)

    # ---- config 4 in small: examples/modelnet_cls/architecture.py:11-81 -----------------------------------------
    ns = exec_reference("examples/modelnet_cls/architecture.py", "ref_modelnet")
    opt = dict(n_filters=32, k=6, act="relu", norm="batch", bias=True, epsilon=0.0, use_stochastic=False, conv="mr",
               n_blocks=4, block="res", use_dilation=True, in_channels=3, n_classes=40, emb_dims=128, dropout=0.5)
    torch.manual_seed(1)
    model = ns["DeepGCN"](types.SimpleNamespace(**opt)).eval()
    randomize_norm(model, gen)
    inputs = torch.rand(3, 3, 160, 1, generator=gen)
    feats, graphs, handles = capture(model)
    with torch.no_grad():
        y = model(inputs)
    for h in handles:
        h.remove()
    outs = {"y": y}
    for i, (f, gph) in enumerate(zip(feats, graphs)):
        outs["feat%d" % i], outs["graph%d" % i] = f, gph
    save("model_mrgcn4", dict(opt, B=3, N=160), {"inputs": inputs}, model.state_dict(), outs)

    # ---- config 3 in small: examples/ogb/ogbn_arxiv/model.py:10-140 ------------------------------------------------
    ns = exec_reference("examples/ogb/ogbn_arxiv/model.py", "ref_arxiv")
    args = dict(num_layers=8, dropout=0.5, block="res+", in_channels=24, hidden_channels=64, num_tasks=10, conv="gen",
                gcn_aggr="softmax_sg", t=0.1, learn_t=False, p=1.0, learn_p=False, y=0.0, learn_y=False,
                msg_norm=False, learn_msg_scale=False, norm="batch", mlp_layers=1)
    torch.manual_seed(2)
    model = ns["DeeperGCN"](types.SimpleNamespace(**args)).eval()
    randomize_norm(model, gen)
    N, E = 700, 6000
    s, d = torch.randint(0, N, (E,), generator=gen), torch.randint(0, N, (E,), generator=gen)
    ei = torch.stack((torch.cat((s, d, torch.arange(N))), torch.cat((d, s, torch.arange(N)))))
    x = torch.randn(N, 24, generator=gen)
    with torch.no_grad():
        y = model(x, ei)
    save("model_deepergcn8", dict(args, N=N), {"x": x, "edge_index": ei.to(torch.int32)}, model.state_dict(), {"y": y})

    # ---- reversible coupling: eff_gcn_modules/rev/memgcn.py:9-52 over the reference GENConv ------------------------------
    sparse = sys.modules["gcn_lib.sparse"]
    src = load_source("eff_gcn_modules/rev/memgcn.py", drop_main=False)
    src = src.split("class InvertibleModuleWrapper")[0] if "class InvertibleModuleWrapper" in src else src
    ns = {"__name__": "ref_memgcn"}
    sys.path.insert(0, os.path.join(ref_shims.REFERENCE_ROOT, "eff_gcn_modules/rev"))
    try:
        exec(compile(src, "memgcn.py", "exec"), ns)
    finally:
        sys.path.pop(0)
    C, group = 64, 2
    torch.manual_seed(3)
    fms = torch.nn.ModuleList(sparse.GENConv(C // group, C // group, aggr="softmax", t=1.0, learn_t=True, msg_norm=True,
                                             learn_msg_scale=True, encode_edge=False, norm="layer", mlp_layers=2)
                              for _ in range(group))
    coupling = ns["GroupAdditiveCoupling"](fms, group=group).eval()
    x = torch.randn(N, C, generator=gen)
    ei = ei[:, torch.randperm(ei.size(1), generator=gen)[:2500]]
    ea = torch.randn(ei.size(1), C, generator=gen) * 0.5      # chunked with x: each GENConv sees (E, C/group) edge features
    with torch.no_grad():
        y = coupling(x, ei, ea)
        x_back = coupling.inverse(y, ei, ea)
    assert torch.allclose(x_back, x, atol=1e-4)
    save("model_revgnn", dict(C=C, group=group, N=N, aggr="softmax", t=1.0, learn_t=True, msg_norm=True,
                              learn_msg_scale=True, norm="layer", mlp_layers=2),
         {"x": x, "edge_index": ei.to(torch.int32), "edge_attr": ea}, coupling.state_dict(), {"y": y, "x_back": x_back})


def sparse_layout_convs():
    """gcn_lib/sparse/torch_vertex.py:91-103, 267-312: MRConv on a random graph (isolated nodes, duplicates) for every
    aggregator, and a ResDynBlock('mr') over equally sized clouds (dilated kNN graph by pairwise distance)."""
    ref_shims.load_reference()
    tv = sys.modules["gcn_lib.sparse.torch_vertex"]
    gen = torch.Generator().manual_seed(21)
    N, E, C = 240, 2000, 24
    ei = torch.stack((torch.randint(0, N - 15, (E,), generator=gen), torch.randint(0, N - 9, (E,), generator=gen)))
    x = torch.randn(N, C, generator=gen)
    outs, sds = {}, {}
    for aggr in ("max", "add", "mean", "min"):
        torch.manual_seed(5)
        conv = tv.MRConv(C, 32, "relu", "batch", True, aggr).eval()
        randomize_norm(conv, gen)
        with torch.no_grad():
            outs["y_" + aggr] = conv(x, ei)
        sds.update({aggr + "." + k: v for k, v in conv.state_dict().items()})
    B, n = 3, 80
    xb = torch.randn(B * n, C, generator=gen)
    batch = torch.arange(B).repeat_interleave(n)
    torch.manual_seed(6)
    blk = tv.ResDynBlock(C, 6, 2, "mr", "relu", "batch", True, res_scale=0.5).eval()
    randomize_norm(blk, gen)
    with torch.no_grad():
        yb, _ = blk(xb, batch)
        eib = blk.body.dilated_knn_graph(xb, batch)
    outs["y_block"], outs["edge_index_block"] = yb, eib.to(torch.int32)
    sds.update({"block." + k: v for k, v in blk.state_dict().items()})
    save("spconv_mr", dict(N=N, C=C, out=32, B=B, n=n, k=6, dilation=2, res_scale=0.5),
         {"x": x, "edge_index": ei.to(torch.int32), "xb": xb, "batch": batch.to(torch.int32)}, sds, outs)


API_DENSE = ("DenseDilated", "DenseDilatedKnnGraph", "DilatedKnnGraph", "MRConv2d", "EdgeConv2d", "GraphConv2d",
             "DynConv2d", "PlainDynBlock2d", "ResDynBlock2d", "DenseDynBlock2d", "BasicConv")
API_SPARSE = ("GENConv", "MsgNorm", "MLP")
API_OPT = dict(n_filters=16, k=4, act="relu", norm="batch", bias=True, epsilon=0.2, stochastic=True, conv="edge",
               n_blocks=3, block="res", in_channels=9, n_classes=13, dropout=0.3)


def reference_api():
    """reference_api.json: the constructor signatures of the public gcn_lib classes ([name, repr(default)] per
    parameter) and the state_dict layout ([key, shape, dtype]) of examples/sem_seg_dense/architecture.py's
    DenseDeepGCN at a small configuration."""
    import inspect
    import json
    dense, sparse = ref_shims.load_reference()

    def sig(cls):
        return [[p.name, repr(p.default)] for p in inspect.signature(cls.__init__).parameters.values()]
    ns = exec_reference("examples/sem_seg_dense/architecture.py", "ref_semseg")
    torch.manual_seed(0)
    model = ns["DenseDeepGCN"](types.SimpleNamespace(**API_OPT))
    sigs = {n: sig(getattr(m, n)) for m, names in ((dense, API_DENSE), (sparse, API_SPARSE)) for n in names}
    sd = [[k, list(v.shape), str(v.dtype)] for k, v in model.state_dict().items()]
    rows = lambda lines: ",\n".join("  " + r for r in lines)      # one class / one tensor per line
    with open(os.path.join(HERE, "reference_api.json"), "w") as fh:
        fh.write('{"signatures": {\n%s\n },\n "dense_deep_gcn_opt": %s,\n "dense_deep_gcn_state_dict": [\n%s\n ]}\n'
                 % (rows("%s: %s" % (json.dumps(n), json.dumps(s)) for n, s in sigs.items()), json.dumps(API_OPT),
                    rows(json.dumps(r) for r in sd)))
    print("wrote reference_api", len(sigs), len(sd))


if __name__ == "__main__":
    main()
    sparse_layout_convs()
    reference_api()
