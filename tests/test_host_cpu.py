"""CPU-side checks: the C-ABI library loads and exports every symbol include/dgcn.h
declares, the drop-in modules keep the reference's constructor signatures and
state_dict keys, and the product path refuses to run without CUDA (no fallback)."""
import ctypes
import os
import re

import pytest
import torch

import golden_util as gu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from deep_gcns_torch_b200 import _native, build
    build.build()
    header = open(os.path.join(ROOT, "include", "dgcn.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = sorted(set(re.findall(r"\b(dgcn_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 15
    handle = ctypes.CDLL(_native.LIB_PATH)
    for name in declared:
        assert hasattr(handle, name), name
    lib = _native.lib()
    assert lib.dgcn_version() >= 100
    assert lib.dgcn_status_string(-2).decode().startswith("request outside")
    # size queries are pure host code: callable without a GPU
    assert lib.dgcn_knn_graph_workspace_bytes(16, 64, 4096, 20) >= 16 * 4096 * 4
    assert lib.dgcn_knn_graph_workspace_bytes(16, 64, 4096, 540) >= 4096 * 4096 * 4
    assert lib.dgcn_csr_build_workspace_bytes(1000, 5000) > 3 * 5000 * 4


def test_struct_layouts_match_header():
    from deep_gcns_torch_b200 import _native
    assert ctypes.sizeof(_native.BasicConvC) == 96
    assert ctypes.sizeof(_native.DilationC) == 32
    assert ctypes.sizeof(_native.GenconvParamsC) == 80
    assert ctypes.sizeof(_native.CsrHubsC) == 40
    assert ctypes.sizeof(_native.GenconvFusionC) == 40
    assert ctypes.sizeof(_native.BlockFusionC) == 40


def test_no_cpu_fallback():
    from deep_gcns_torch_b200.gcn_lib import dense as D, sparse as S
    x = torch.randn(1, 4, 16, 1)
    with pytest.raises(RuntimeError, match="CUDA"):
        D.DynConv2d(4, 4, 3)(x)
    with pytest.raises(RuntimeError, match="CUDA"):
        D.DenseDilatedKnnGraph(3)(x)
    with pytest.raises(RuntimeError, match="CUDA"):
        S.GENConv(4, 4)(torch.randn(5, 4), torch.zeros((2, 3), dtype=torch.long))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "deep_gcns_torch_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, f


@pytest.mark.parametrize("name", [n for n in gu.names("dense_") if "grid" not in n])
def test_dense_state_dict_compat(name):
    from deep_gcns_torch_b200.gcn_lib import dense as D
    c = gu.load(name)
    m = c.meta
    if "static" in name:
        mod = D.GraphConv2d(m["in_channels"], m["out_channels"], m["conv"], m["act"], m["norm"], m["bias"])
    else:
        mod = D.DynConv2d(m["in_channels"], m["out_channels"], m["k"], m["dilation"], m["conv"], m["act"],
                          m["norm"], m["bias"])
    own = mod.state_dict()
    assert list(own.keys()) == list(c.sd.keys())
    assert all(tuple(own[k].shape) == tuple(c.sd[k].shape) and own[k].dtype == c.sd[k].dtype for k in own)
    mod.load_state_dict(c.sd, strict=True)


@pytest.mark.parametrize("name", gu.names("sparse_"))
def test_sparse_state_dict_compat(name):
    from deep_gcns_torch_b200.gcn_lib import sparse as S
    c = gu.load(name)
    m = dict(c.meta)
    in_dim, emb_dim = m.pop("in_dim"), m.pop("emb_dim")
    m.pop("N")
    mod = S.GENConv(in_dim, emb_dim, **m)
    own = mod.state_dict()
    assert list(own.keys()) == list(c.sd.keys())
    assert all(tuple(own[k].shape) == tuple(c.sd[k].shape) for k in own)
    mod.load_state_dict(c.sd, strict=True)
    assert isinstance(getattr(mod, "t", 1.0), (float, torch.nn.Parameter))


def test_signatures_match_live_reference():
    """Constructor signatures of the drop-in classes and the state_dict layout of a model stack built on them against
    the reference's, as stored by gen_golden_models.py's reference_api (tests/golden/reference_api.json)."""
    import inspect
    import json
    from bench_models import ResGCN28
    from deep_gcns_torch_b200.gcn_lib import dense as D, sparse as S
    with open(os.path.join(gu.GOLDEN_DIR, "reference_api.json")) as fh:
        api = json.load(fh)
    assert len(api["signatures"]) == 14
    for name, ref in api["signatures"].items():
        mine = getattr(S if name in ("GENConv", "MsgNorm", "MLP") else D, name)
        assert [[p.name, repr(p.default)] for p in inspect.signature(mine.__init__).parameters.values()] == ref, name
    # the reference's sem_seg_dense DenseDeepGCN, assembled from the drop-in classes (bench_models.py restates it)
    opt = api["dense_deep_gcn_opt"]
    assert (opt["block"], opt["conv"], opt["act"], opt["norm"], opt["bias"], opt["stochastic"], opt["epsilon"],
            opt["dropout"]) == ("res", "edge", "relu", "batch", True, True, 0.2, 0.3)
    mine = ResGCN28(D, opt["in_channels"], opt["n_classes"], opt["k"], opt["n_filters"], opt["n_blocks"])
    theirs = {k: torch.zeros(shape, dtype=getattr(torch, dt.split(".")[1])) for k, shape, dt in
              api["dense_deep_gcn_state_dict"]}
    assert list(mine.state_dict().keys()) == list(theirs.keys())
    assert all(v.dtype == theirs[k].dtype for k, v in mine.state_dict().items())
    mine.load_state_dict(theirs, strict=True)


def test_bench_line_carries_every_contract_key():
    """Static check of bench.py's JSON line (no GPU): the dict literal assembled in run_native, evaluated
    with stand-in measurements, has every key of the bench contract and consistent derived values."""
    import ast
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    path = os.path.join(root, "bench.py")
    tree = ast.parse(open(path).read())
    g = {"__file__": path, "__name__": "bench_static"}
    top = [n for n in tree.body if isinstance(n, (ast.Assign, ast.Import, ast.ImportFrom))]
    exec(compile(ast.Module(top, []), path, "exec"), g)
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "run_native")
    lit = next(n.value for n in ast.walk(fn) if isinstance(n, ast.Assign) and isinstance(n.targets[0], ast.Name)
               and n.targets[0].id == "out" and isinstance(n.value, ast.Dict))

    class Args:
        steps, warmup = 20, 1

    loc = dict(world=2, args=Args, ms=11.4, ms_e2e=12.7, clk={"sm_mhz": 1965.0}, achieved=220.0, peak=6563.9,
               traffic=72000000, peak_src="measured", kernel_ms=0.507, tensor_peak=1691.8, sm_max=1965.0,
               hbm_achieved=66.0, tensor_flop=1.1e11, numa={"numa_node": 0})
    out = eval(compile(ast.Expression(lit), path, "eval"), g, loc)
    json.dumps(out)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
        assert key in out, key
    assert out["warmup"] >= 3 and out["n_gpus"] == 2 and out["scaling"] == "weak" and out["vs_baseline"] is None
    assert set(("bound", "achieved", "peak", "unit", "frac", "traffic")) <= set(out["roofline"])
    assert out["roofline"]["bound"] in ("hbm", "tensor") and out["roofline"]["unit"] == "TFLOP/s"
    assert abs(out["roofline"]["frac"] - 220.0 / 1691.8) < 1e-9 and out["roofline"]["hbm"]["unit"] == "GB/s"
    assert set(("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")) <= set(out["e2e"])
    assert "workload" in out["config"] and "model" not in out["config"]
    edges = 16 * 4096 * 20
    assert abs(out["value"] - edges * 2 * 20 / 11.4e-3) < 1.0          # whole-job aggregate over both ranks
    assert out["gpu_launches"] > 0
