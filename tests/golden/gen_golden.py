"""Generates the committed golden vectors under tests/golden/*.npz by running
the UNMODIFIED reference modules (/root/reference/gcn_lib, loaded through
oracle/ref_shims.py) on seeded synthetic inputs.  The reference has no tests
or fixtures of its own (SURVEY.md 4), so these vectors are what pins parity.

    python tests/golden/gen_golden.py        # needs /root/reference

Each file holds: `in.*` inputs, `sd.*` the reference module's state_dict,
`out.*` reference outputs, `meta` (JSON: constructor arguments).
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_shims  # noqa: E402


def save(name, meta, ins, sd, outs):
    blob = {"meta": np.array(json.dumps(meta))}
    for k, v in ins.items():
        blob["in." + k] = v.numpy()
    for k, v in sd.items():
        blob["sd." + k] = v.numpy()
    for k, v in outs.items():
        blob["out." + k] = v.numpy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **blob)
    print("wrote", name, {k: tuple(v.shape) for k, v in outs.items()})


def randomize_norm(mod, gen):
    """Non-trivial affine + running stats (incl. negative gamma) so eval-mode
    BN is a real test of conv -> act -> norm -> max ordering."""
    for m in mod.modules():
        if isinstance(m, (torch.nn.BatchNorm2d, torch.nn.BatchNorm1d)):
            c = m.num_features
            m.weight.data = torch.randn(c, generator=gen) * 0.7 + 0.3
            m.bias.data = torch.randn(c, generator=gen) * 0.2
            m.running_mean.data = torch.randn(c, generator=gen) * 0.3
            m.running_var.data = torch.rand(c, generator=gen) + 0.4
        if isinstance(m, torch.nn.Conv2d) and m.bias is not None:
            m.bias.data = torch.randn(m.bias.shape, generator=gen) * 0.1


def dense_cases(dense):
    # (name, B, Cin, Cout, N, k, d, conv, act, norm, bias, training, input kind)
    cases = [
        ("dense_c1_edge", 2, 32, 32, 1024, 16, 1, "edge", "relu", "batch", True, False, "randn"),
        ("dense_c1_mr", 2, 32, 32, 1024, 16, 1, "mr", "relu", "batch", True, False, "randn"),
        ("dense_edge_dil3_leaky_batch", 2, 8, 24, 256, 4, 3, "edge", "leakyrelu", "batch", True, False, "randn"),
        ("dense_edge_dil2_prelu_none", 3, 6, 16, 200, 5, 2, "edge", "prelu", None, False, False, "randn"),
        ("dense_mr_dil4_leaky_batch", 2, 16, 48, 320, 9, 4, "mr", "leakyrelu", "batch", True, False, "rand"),
        ("dense_edge_train_bn", 2, 12, 20, 192, 6, 2, "edge", "relu", "batch", True, True, "randn"),
        ("dense_mr_train_bn", 2, 12, 20, 192, 6, 2, "mr", "relu", "batch", True, True, "randn"),
        ("dense_head_c3_edge", 2, 3, 64, 512, 20, 1, "edge", "relu", "batch", True, False, "rand"),
        ("dense_edge_bigk", 1, 16, 16, 640, 20, 8, "edge", "relu", "batch", True, False, "randn"),
    ]
    for (name, B, ci, co, N, k, d, conv, act, norm, bias, training, kind) in cases:
        gen = torch.Generator().manual_seed(0)
        torch.manual_seed(0)
        mod = dense.DynConv2d(ci, co, k, d, conv, act, norm, bias)
        randomize_norm(mod, gen)
        x = (torch.randn if kind == "randn" else torch.rand)(B, ci, N, 1, generator=gen)
        mod.train(training)
        sd_before = {kk: vv.clone() for kk, vv in mod.state_dict().items()}
        extra = {}
        with torch.no_grad():
            ei = mod.dilated_knn_graph(x)
            full = dense.dense_knn_matrix(x, k * d)
            y = mod(x)          # builds the same graph again internally
            if not training:
                assert torch.equal(y, dense.GraphConv2d.forward(mod, x, ei))
            else:               # running statistics after exactly ONE training forward
                bn = mod.gconv.nn[2]
                extra = {"running_mean": bn.running_mean.clone(), "running_var": bn.running_var.clone(),
                         "num_batches_tracked": bn.num_batches_tracked.clone()}
        meta = dict(B=B, in_channels=ci, out_channels=co, N=N, k=k, dilation=d, conv=conv, act=act,
                    norm=norm, bias=bias, training=training)
        save(name, meta, {"x": x}, sd_before,
             dict(extra, y=y, nn_idx=ei[0].to(torch.int32), nn_idx_full=full[0].to(torch.int32),
                  center_idx=ei[1].to(torch.int32)))

    # exact-arithmetic kNN case: coordinates on a 1/8 grid so every fp32
    # evaluation order gives the same distances; ties are frequent on purpose.
    gen = torch.Generator().manual_seed(1)
    x = torch.randint(-16, 17, (2, 4, 128, 1), generator=gen).float() / 8
    full = dense.dense_knn_matrix(x, 128)
    xt = x.squeeze(-1).transpose(2, 1)
    dist = dense.pairwise_distance(xt)
    save("dense_knn_grid_ties", dict(B=2, C=4, N=128, K=128), {"x": x}, {},
         {"nn_idx_full": full[0].to(torch.int32), "dist": dist})

    # arbitrary centre indices through the static GraphConv2d API
    gen = torch.Generator().manual_seed(2)
    torch.manual_seed(2)
    for conv in ("edge", "mr"):
        mod = dense.GraphConv2d(10, 14, conv, "relu", "batch", True).eval()
        randomize_norm(mod, gen)
        x = torch.randn(2, 10, 96, 1, generator=gen)
        ei = torch.randint(0, 96, (2, 2, 96, 7), generator=gen)
        with torch.no_grad():
            y = mod(x, ei)
        save("dense_static_%s_arbitrary_centres" % conv,
             dict(in_channels=10, out_channels=14, conv=conv, act="relu", norm="batch", bias=True),
             {"x": x, "edge_index": ei.to(torch.int32)}, mod.state_dict(), {"y": y})


def sparse_cases(sparse):
    gen = torch.Generator().manual_seed(0)
    N, E, C = 300, 3000, 32
    src = torch.randint(0, N - 20, (E,), generator=gen)       # last 20 nodes isolated as sources
    dst = torch.randint(0, N - 10, (E,), generator=gen)       # last 10 nodes have no in-edges
    dst[:400] = 7                                             # one hub row
    ei = torch.stack((torch.cat([src, torch.arange(0, 50)]), torch.cat([dst, torch.arange(0, 50)])), 0)
    x = torch.randn(N, C, generator=gen)
    ea = torch.randn(ei.size(1), 5, generator=gen)
    cfgs = [
        ("softmax_sg", dict(aggr="softmax_sg", t=0.1, mlp_layers=1)),
        ("softmax_learn_t", dict(aggr="softmax", t=0.7, learn_t=True, msg_norm=True, mlp_layers=2)),
        ("softmax_fixed", dict(aggr="softmax", t=1.0, mlp_layers=1, norm="layer")),
        ("softmax_sum", dict(aggr="softmax_sum", t=0.5, learn_t=True, y=0.3, learn_y=True, mlp_layers=1)),
        ("power", dict(aggr="power", p=2.0, learn_p=True, msg_norm=True, learn_msg_scale=True, mlp_layers=1)),
        ("power_sum", dict(aggr="power_sum", p=3.0, y=-0.4, learn_y=True, mlp_layers=2)),
        ("add", dict(aggr="add", mlp_layers=1)),
        ("mean", dict(aggr="mean", mlp_layers=1)),
        ("max", dict(aggr="max", msg_norm=True, mlp_layers=1)),
        ("softmax_edge_attr", dict(aggr="softmax", t=1.0, encode_edge=True, edge_feat_dim=5, mlp_layers=1)),
    ]
    for name, kw in cfgs:
        torch.manual_seed(0)
        mod = sparse.GENConv(C, C if "edge" not in name else 40, **kw).eval()
        randomize_norm(mod, gen)
        if mod.msg_norm is not None:
            mod.msg_norm.msg_scale.data.fill_(0.8)
        use_ea = kw.get("encode_edge", False)
        with torch.no_grad():
            y = mod(x, ei, ea if use_ea else None)
            m = mod.propagate(ei, x=x, edge_attr=mod.edge_encoder(ea) if use_ea else None)
        ins = {"x": x, "edge_index": ei.to(torch.int32)}
        if use_ea:
            ins["edge_attr"] = ea
        save("sparse_" + name, dict(in_dim=C, emb_dim=int(y.shape[1]), N=N, **kw), ins,
             mod.state_dict(), {"y": y, "m": m})


def sparse_edge_cases():
    """gcn_lib/sparse/torch_edge.py (knn='matrix'): flattened, globally numbered kNN graphs of equally
    sized clouds; regular and stochastic dilation (the latter under a fixed CPU RNG seed)."""
    te = sys.modules["gcn_lib.sparse.torch_edge"]
    gen = torch.Generator().manual_seed(3)
    B, n, C = 4, 96, 7
    x = torch.randn(B * n, C, generator=gen)
    batch = torch.arange(B).repeat_interleave(n)
    outs = {"knn_k9": te.knn_graph_matrix(x, 9, batch),
            "dilated_k5_d2": te.DilatedKnnGraph(5, 2)(x, batch),
            "single_cloud_k6_d3": te.DilatedKnnGraph(6, 3)(x[:n], None if False else torch.zeros(n, dtype=torch.long))}
    sto = te.DilatedKnnGraph(5, 3, True, 1.0).train()
    torch.manual_seed(11)
    outs["stochastic_k5_d3_seed11"] = sto(x, batch)
    full = te.knn_graph_matrix(x, 15, batch)
    dil = te.Dilated(5, 3, True, 1.0).train()
    torch.manual_seed(12)
    outs["dilated_module_seed12"] = dil(full)
    save("spgraph_knn_matrix", dict(B=B, n=n, C=C), {"x": x, "batch": batch.to(torch.int32)}, {},
         {k: v.to(torch.int32) for k, v in outs.items()})


PIN_DENSE_SHAPES = [(1, 5, 77, 3, 2), (3, 20, 130, 7, 1), (2, 3, 64, 8, 8)]      # (B, C, N, k, dilation)
PIN_AGGRS = ("softmax", "softmax_sg", "softmax_sum", "power", "power_sum", "add", "mean", "max")
PIN_GRAPHS = ((4, 1), (3, 4))                                                     # (k, dilation)


def pin_cases(dense, sparse):
    """Small odd shapes through the reference's default-initialised modules (no randomize_norm): the dense kNN
    matrix, DynConv2d(C, 9, k, d, conv, 'leakyrelu', 'batch') in eval, GENConv(12, 12) for every aggregator with
    learnable t and message norm, and the sparse DilatedKnnGraph over three clouds."""
    te = sys.modules["gcn_lib.sparse.torch_edge"]
    g = torch.Generator().manual_seed(11)
    ins, sd, outs = {}, {}, {}
    for s, (B, C, N, k, d) in enumerate(PIN_DENSE_SHAPES):
        x = torch.randn(B, C, N, 1, generator=g)
        ins["x%d" % s] = x
        outs["knn%d" % s] = dense.dense_knn_matrix(x, k * d).to(torch.int32)
        for conv in ("edge", "mr"):
            torch.manual_seed(3)
            mod = dense.DynConv2d(C, 9, k, d, conv, "leakyrelu", "batch", True).eval()
            with torch.no_grad():
                outs["y%d_%s" % (s, conv)] = mod(x)
            sd.update({"s%d_%s.%s" % (s, conv, kk): vv for kk, vv in mod.state_dict().items()})
    ins["xs"] = torch.randn(90, 12, generator=g)
    ins["edge_index"] = torch.randint(0, 90, (2, 500), generator=g).to(torch.int32)
    for aggr in PIN_AGGRS:
        torch.manual_seed(4)
        mod = sparse.GENConv(12, 12, aggr=aggr, t=0.3, learn_t=True, p=2.0, y=0.2, msg_norm=True).eval()
        with torch.no_grad():
            outs["gen_" + aggr] = mod(ins["xs"], ins["edge_index"].long())
        sd.update({"%s.%s" % (aggr, kk): vv for kk, vv in mod.state_dict().items()})
    ins["xg"] = torch.randn(3 * 50, 6, generator=g)
    ins["batch"] = torch.arange(3).repeat_interleave(50).to(torch.int32)
    for k, d in PIN_GRAPHS:
        outs["graph_k%d_d%d" % (k, d)] = te.DilatedKnnGraph(k, d)(ins["xg"], ins["batch"].long()).to(torch.int32)
    save("pin_random_shapes", dict(dense=PIN_DENSE_SHAPES, act="leakyrelu", norm="batch", aggrs=PIN_AGGRS,
                                   graphs=PIN_GRAPHS), ins, sd, outs)


if __name__ == "__main__":
    torch.set_num_threads(8)
    dense, sparse = ref_shims.load_reference()
    dense_cases(dense)
    sparse_cases(sparse)
    sparse_edge_cases()
    pin_cases(dense, sparse)
