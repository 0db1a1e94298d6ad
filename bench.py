#!/usr/bin/env python
"""Headline benchmark: edges/s of one DynConv2d forward (dilated kNN graph + EdgeConv,
B=16 N=4096 k=20 C=64 - BASELINE.json's metric shape) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of 16 synthetic clouds
(1,310,720 edges).  Multi-GPU: the batch dimension is sharded, every rank owns its
own 16 clouds (weak scaling, no data-path collective - clouds are independent,
SURVEY.md 8e).  Prints ONE JSON line (rank 0; file descriptor 1 is pointed at stderr
for everything else - NCCL's version banner, warnings).  The K timed steps are
enqueued behind a ~2 ms spin kernel and bracketed by CUDA events: a step is ~0.25 ms
of GPU time, so the host's first-launch latency after the synchronize would otherwise
be several percent of a 20-step region.

`--dump-outputs DIR` writes what the K-th timed step returned, DynConv2d's (16, 64, 4096, 1) fp32 output (16.8 MB),
as DIR/y.npy once all timing is done; inputs and weights are seeded, so the file depends only on the arguments and
on the build (`--impl reference`: its own last step, 4 clouds).

`--impl reference` times the reference's CPU algorithm (the oracle port: the
reference is pure Python/torch, there is nothing to compile into oracle/_ref) on the
host cores of the box, each step a bounded sample (4 of the 16 clouds), with the
thread count that is fastest on this box (the reference's N^2 elementwise passes are
memory bound: all 128 hardware threads are slower than 16-32).

At N = 1 the line also carries `gpu_reference` (the reference's op sequence - oracle
port - running as torch-eager CUDA kernels on the same B200, the comparison target of
north_star's ">= 10x the reference GPU path") and `sustained` (the same step looped
for >= 2 s with clocks sampled).  At N > 1 `extra` carries the node-partitioned
GENConv stack on the products-shaped graph (`sparse_halo`) and one data-parallel
MRGCN-28 training step (`ddp_mrgcn`), each with its parity check (bench_multigpu.py).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B, C, N, K_NEIGH, DIL = 16, 64, 4096, 20, 1
EDGES_PER_STEP = B * N * K_NEIGH
# SURVEY.md 8d: compulsory bytes per edge with the graph fused (read x once, write y once)
ALGO_BYTES_PER_EDGE = (C + C) * 4.0 / K_NEIGH            # 25.6 B
# fp32 work per edge: distance contraction 2*N*C/k + factorised MLP 2*2C*C/k (SURVEY.md 8d)
FLOPS_PER_EDGE = 2.0 * N * C / K_NEIGH + 2.0 * 2 * C * C / K_NEIGH
N_ROTATE = 8                                             # 8 x 16.8 MB inputs = 134 MB > 126 MB L2
WORKLOAD = "DynConv2d(64,64,k=20,d=1,edge,relu,batch).eval() fwd, x=randn(16,64,4096,1)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--sustained-seconds", type=float, default=2.0, help="length of the sustained loop (N=1)")
    ap.add_argument("--no-extra", action="store_true", help="skip the multi-GPU extra blocks (N>1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output of the last timed step as DIR/y.npy (float32; rank 0's clouds at N>1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(directory, arrays):
    """{name: array} -> directory/<name>.npy.  The inputs are seeded, so two builds run with the same arguments can be
    compared output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def bind_to_gpu_numa_node(index):
    """Pin this process (and therefore the pinned host buffers it is about to allocate, first touch) to the
    CPUs of the NUMA node the GPU hangs off.  Returns a description for the JSON line."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(index).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:                      # nvml prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as fh:
            node = int(fh.read().strip())
        if node < 0:
            return {"numa_node": None, "note": "single NUMA node"}
        with open("/sys/devices/system/node/node%d/cpulist" % node) as fh:
            cpus = set()
            for part in fh.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as exc:                                  # binding is an optimisation, never a failure
        return {"numa_node": None, "note": "not bound: %s" % type(exc).__name__}


def best_cpu_threads(run, x, candidates, budget_s):
    """Thread count (of `candidates`) at which the oracle layer is fastest on this box, (threads, seconds/run)."""
    import torch
    best = None
    for th in candidates:
        torch.set_num_threads(th)
        run(x)
        t0 = time.perf_counter()
        n = 0
        while n < 1 or (time.perf_counter() - t0 < budget_s / len(candidates) and n < 3):
            run(x)
            n += 1
        dt = (time.perf_counter() - t0) / n
        if best is None or dt < best[1]:
            best = (th, dt)
    torch.set_num_threads(best[0])
    return best


def thread_candidates():
    avail = len(os.sched_getaffinity(0))
    return sorted({t for t in (8, 16, 32, 64, avail) if t <= avail})


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return (float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", float(p.get("sm_max_mhz", 1965.0)),
                float(p.get("bf16_tflops", 1590.0)))
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)", 1965.0, 1590.0


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region.

    The timed region of the default run lasts ~10 ms, far below nvidia-smi's 100-200 ms loop period, so the
    samples come from NVML directly (the library nvidia-smi itself reads: `clocks.sm`, `clocks.max.sm`,
    `clocks_event_reasons.*`), polled from a thread every ~2 ms between __enter__ and __exit__; the
    nvidia-smi loop of the profiling recipe is the fallback when pynvml is unavailable."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    # nvmlClocksEventReasons bits
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.samples, self.max_mhz, self.reasons = [], 0.0, set()
        self.nvml, self.handle, self.stop = None, None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            handle = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
                handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml, self.handle = pynvml, handle
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _poll_once(self):
        nv = self.nvml
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
        try:
            mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        for name, bit in self.REASONS.items():
            if mask & bit:
                self.reasons.add(name)

    def _poll(self):
        while not self.stop.is_set():
            try:
                self._poll_once()
            except Exception:
                return
            time.sleep(0.002)      # a poll holds the GIL for tens of microseconds: keep it rare next to a 0.26 ms step

    def __enter__(self):
        self.stop.clear()
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return self
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def __exit__(self, *exc):
        if self.nvml is not None:
            try:
                self._poll_once()            # the GPU is still inside (or just leaving) the timed region
            except Exception:
                pass
            self.stop.set()
            self.thread.join(timeout=2)
            return
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = list(self.samples), self.max_mhz, set(self.reasons)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = max(mx, float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi -lms 100"}


def oracle_layer(threads):
    """The reference algorithm (oracle port) and its parameters for the headline layer."""
    import torch
    from oracle import dense as od
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    conv = torch.nn.Conv2d(2 * C, C, 1)
    torch.nn.init.kaiming_normal_(conv.weight)
    p = {"weight": conv.weight.detach(), "bias": torch.zeros(C),
         "norm": {"weight": torch.ones(C), "bias": torch.zeros(C), "running_mean": torch.zeros(C),
                  "running_var": torch.ones(C)}}

    def run(x):
        with torch.no_grad():
            return od.dyn_conv(x, p, K_NEIGH, DIL, "edge", "relu", "batch")
    return run


def cpu_sample(gen_seed=0, clouds=4):
    import torch
    g = torch.Generator().manual_seed(gen_seed)
    return torch.randn(clouds, C, N, 1, generator=g)


def run_reference(args):
    """--impl reference: reference CPU path, all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    run = oracle_layer(len(os.sched_getaffinity(0)))
    clouds = 4
    x = cpu_sample(clouds=clouds)
    edges = clouds * N * K_NEIGH
    threads, _ = best_cpu_threads(run, x, thread_candidates(), 20.0)   # untimed calibration (part of the warm-up)
    for _ in range(max(args.warmup, 1)):
        run(x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        y = run(x)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"y": y.numpy()})
    value = edges * args.steps / dt
    sample = ("%d of the %d clouds per step (clouds are independent), %d steps, %d threads = fastest of %s on the "
              "%d available" % (clouds, B, args.steps, threads, thread_candidates(), len(os.sched_getaffinity(0))))
    print(json.dumps({
        "impl": "reference", "metric": "edges/sec EdgeConv fwd (B=16,N=4096,k=20,C=64)", "value": value,
        "unit": "edges/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "edges/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def gpu_reference_block(dev, steps, warmup):
    """The reference's own op sequence (oracle port of gcn_lib/dense/torch_edge.py:32-58 + torch_vertex.py:31-35 +
    torch_nn.py:48-58, the code examples/sem_seg_dense/architecture.py:99-109 times) as torch-eager CUDA kernels on
    this GPU: fp32, TF32 off, same layer, same inputs.  A baseline leg - none of this repo's kernels run here."""
    import torch
    from oracle import dense as od
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(0)
    conv = torch.nn.Conv2d(2 * C, C, 1)
    torch.nn.init.kaiming_normal_(conv.weight)
    p = {"weight": conv.weight.detach().to(dev), "bias": torch.zeros(C, device=dev),
         "norm": {"weight": torch.ones(C, device=dev), "bias": torch.zeros(C, device=dev),
                  "running_mean": torch.zeros(C, device=dev), "running_var": torch.ones(C, device=dev)}}
    g = torch.Generator().manual_seed(1000)
    xs = [torch.randn(B, C, N, 1, generator=g).to(dev) for _ in range(2)]
    with torch.no_grad():
        for i in range(max(warmup, 2)):
            od.dyn_conv(xs[i & 1], p, K_NEIGH, DIL, "edge", "relu", "batch")
        torch.cuda.synchronize()
        beg, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        beg.record()
        for i in range(steps):
            od.dyn_conv(xs[i & 1], p, K_NEIGH, DIL, "edge", "relu", "batch")
        end.record()
        torch.cuda.synchronize()
    ms = beg.elapsed_time(end) / steps
    del xs
    torch.cuda.empty_cache()
    return {"value": EDGES_PER_STEP / (ms * 1e-3), "unit": "edges/s", "ms_per_step": ms, "steps": steps,
            "what": "reference op sequence (oracle port) as torch-eager CUDA kernels on the same GPU, fp32, TF32 off, "
                    "inputs resident, peak memory ~5 GB (B x N x N distance matrix + gathered edge features)"}


def sparse_aggregate_block(dev, steps=10):
    """GENConv softmax aggregate (message + online softmax + residual, one fused kernel) on a synthetic
    ogbn-products-shaped CSR (N = 2,449,029, E = 61,859,140 uniform edges, C = 128; x = 1.25 GB >> L2), against the
    gather-model HBM roofline of SURVEY.md 8d: 4C+4 B/edge + (8C+4) B/node.  Target (north_star): >= 60 % of the
    measured HBM peak.  L2 is flushed between iterations."""
    import torch
    from deep_gcns_torch_b200 import _native
    N, E, C = 2449029, 61859140, 128
    g = torch.Generator(device=dev).manual_seed(0)
    ei = torch.stack((torch.randint(0, N, (E,), generator=g, device=dev), torch.randint(0, N, (E,), generator=g, device=dev)))
    x = torch.randn(N, C, generator=g, device=dev)
    csr = _native.csr_build(ei, N)
    del ei
    prm, _keep = _native.genconv_params("softmax_sg", 0.1, 1.0, 0.0, 1e-7, None, add_residual=True)
    out = torch.empty_like(x)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for _ in range(3):
        _native.genconv_aggregate(x, x, csr, prm, out=out)
    times = []
    beg, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(steps):
        flush.zero_()
        beg.record()
        _native.genconv_aggregate(x, x, csr, prm, out=out)
        end.record()
        torch.cuda.synchronize()
        times.append(beg.elapsed_time(end))
    times.sort()
    ms = times[len(times) // 2]
    peak = peaks()[0]
    gather_bytes = E * (4 * C + 4) + N * (8 * C + 4)
    res = {"workload": "GENConv aggregate softmax_sg t=0.1, N=%d E=%d C=%d (products-shaped, uniform)" % (N, E, C),
           "ms": ms, "edges_per_s": E / (ms * 1e-3), "steps": steps,
           "roofline": {"bound": "hbm", "achieved": gather_bytes / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": gather_bytes / (ms * 1e-3) / 1e9 / peak, "bytes_per_launch": gather_bytes,
                        "model": "gather model: 4C+4 B/edge + (8C+4) B/node (SURVEY.md 8d); ncu dram bytes of the same "
                                 "launch: profiles/r02_aggregate_products_ncu.json"}}
    del x, out, flush, csr
    torch.cuda.empty_cache()
    return res


def _claim_stdout():
    """Keep stdout to the ONE JSON line: file descriptor 1 is pointed at stderr for the whole run (NCCL prints its
    version banner to fd 1 from C, torch prints warnings), the JSON line is written to a saved copy of the real stdout."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, "w")


def run_native(args):
    import torch
    import torch.distributed as dist
    json_out = _claim_stdout()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)          # before the pinned buffers exist: they are first-touched locally
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line (NCCL's version banner)
        dist.init_process_group("nccl", device_id=dev)
    from deep_gcns_torch_b200 import _native
    from deep_gcns_torch_b200.gcn_lib import dense as D

    torch.manual_seed(0)
    mod = D.DynConv2d(C, C, K_NEIGH, DIL, "edge", "relu", "batch", True).to(dev).eval()
    g = torch.Generator().manual_seed(1000 + rank)
    host = [torch.randn(B, C, N, 1, generator=g).pin_memory() for _ in range(N_ROTATE)]
    xs = [h.to(dev) for h in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident-input throughput ("value") --------------------------------------------
    with torch.no_grad():
        for i in range(max(args.warmup, 3)):
            mod(xs[i % N_ROTATE])
        barrier()
        _native.kernel_timing(True)
        _native.kernel_timing_read("knn")
        beg, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local) as clocks:
            barrier()
            # ~2 ms spin kernel ahead of the first event: the host enqueues the first steps behind it, so the K timed
            # steps run back to back as they do in steady state (a step is ~0.25 ms of GPU time against ~0.2 ms of
            # host-side launch work: without the head start the first-launch latency after the synchronize is 5-15 %
            # of a 20-step region; the `sustained` block below is the same loop over ~2 s without any of this)
            torch.cuda._sleep(4_000_000)
            beg.record()
            for i in range(args.steps):
                y = mod(xs[i % N_ROTATE])
            end.record()
            barrier()
        ms = beg.elapsed_time(end)
        knn_ms, knn_n = _native.kernel_timing_read("knn")
        _native.kernel_timing(False)
        last_step = {"y": y.cpu().numpy()} if args.dump_outputs and rank == 0 else None
        del y

        # ---- end to end: pinned host input -> device -> DynConv2d -> pinned host result -------------
        # Every step copies ITS input from pinned host memory and ITS result back, inside the timed
        # region; the copies run on their own streams so step i+1's upload and step i-1's download
        # overlap step i's kernels (what a serving loop around the public module call does).
        h2d, d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        cur = torch.cuda.current_stream(dev)
        xin = [torch.empty_like(xs[0]) for _ in range(2)]
        up_done = [torch.cuda.Event() for _ in range(2)]
        comp_done = [torch.cuda.Event() for _ in range(2)]
        host_outs = [torch.empty(B, C, N, 1).pin_memory() for _ in range(2)]

        def e2e_loop(n):
            for i in range(n):
                sl = i & 1
                with torch.cuda.stream(h2d):
                    h2d.wait_event(comp_done[sl])            # buffer free: step i-2 has consumed it
                    xin[sl].copy_(host[i % N_ROTATE], non_blocking=True)
                    up_done[sl].record(h2d)
                cur.wait_event(up_done[sl])
                y = mod(xin[sl])                             # the public API call
                comp_done[sl].record(cur)
                y.record_stream(d2h)
                with torch.cuda.stream(d2h):
                    d2h.wait_event(comp_done[sl])
                    host_outs[sl].copy_(y, non_blocking=True)
        e2e_loop(4)
        barrier()
        b2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with clocks:                                     # the end-to-end region is sampled as well
            b2.record(cur)
            h2d.wait_event(b2)
            e2e_loop(args.steps)
            cur.wait_stream(d2h)
            cur.wait_stream(h2d)
            e2.record(cur)
            barrier()
        ms_e2e = b2.elapsed_time(e2)

        # ---- sustained: the same resident-input step looped for >= sustained_seconds (N = 1) --------------
        sustained = None
        if world == 1 and args.sustained_seconds > 0:
            n_sus = max(args.steps, int(args.sustained_seconds / max(ms / args.steps * 1e-3, 1e-6)) + 1)
            sb_, se_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with ClockSampler(local) as sclk:
                sb_.record()
                for i in range(n_sus):
                    mod(xs[i % N_ROTATE])
                se_.record()
                torch.cuda.synchronize()
            ms_sus = sb_.elapsed_time(se_)
            sustained = {"value": EDGES_PER_STEP * n_sus / (ms_sus * 1e-3), "unit": "edges/s", "steps": n_sus,
                         "seconds": ms_sus * 1e-3, "ms_per_step": ms_sus / n_sus, "clocks": sclk.summary()}

    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])

    # ---- N = 1: the sparse hot kernel against its HBM roofline on the products-shaped CSR (outside the timed regions) ----
    extra = None
    if world == 1 and not args.no_extra:
        try:
            extra = {"sparse_aggregate": sparse_aggregate_block(dev)}
        except Exception as exc:
            extra = {"sparse_aggregate": {"error": "%s: %s" % (type(exc).__name__, exc)}}
    # ---- multi-GPU blocks (outside the headline's timed regions): config 5 and config 4 ---------------------
    if world > 1 and not args.no_extra:
        import bench_multigpu as bm
        extra = {}
        for name, fn in (("sparse_halo", bm.sparse_halo_block), ("ddp_mrgcn", bm.ddp_mrgcn_block)):
            try:
                extra[name] = fn(dev, rank, world)
            except Exception as exc:                     # a failing extra block must not take the headline line down
                import traceback
                extra[name] = {"error": "%s: %s" % (type(exc).__name__, exc), "trace": traceback.format_exc()[-1500:],
                               "parity_ok": False}
                try:
                    dist.barrier()
                except Exception:
                    pass
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src, sm_max, tensor_peak = peaks()
    kernel_ms = knn_ms / max(knn_n, 1)
    hbm_achieved = EDGES_PER_STEP * ALGO_BYTES_PER_EDGE / (kernel_ms * 1e-3) / 1e9
    tensor_flop = 2.0 * B * N * N * (3 * C + 16)     # 3 split products hi*hi, hi*mid, mid*hi over C channels + one K=16 block folding -|x_j|^2/2
    achieved = tensor_flop / (kernel_ms * 1e-3) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as fh:
            traffic = json.load(fh).get("knn_tc4_kernel")
    clk = clocks.summary()
    out = {
        "metric": "edges/sec EdgeConv fwd (B=16,N=4096,k=20,C=64)",
        "value": EDGES_PER_STEP * world * args.steps / (ms * 1e-3),
        "unit": "edges/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "edges_per_step_per_gpu": EDGES_PER_STEP, "parallelism": "batch-sharded x%d" % world,
                   "l2": "inputs rotate over %d distinct 16.8 MB batches (134 MB > 126 MB L2)" % N_ROTATE,
                   "queue": "the K timed steps are enqueued behind a ~2 ms spin kernel (device-side throughput; CUDA events "
                            "bracket exactly the K steps)",
                   "host_binding": numa},
        "e2e": {"value": EDGES_PER_STEP * world * args.steps / (ms_e2e * 1e-3), "unit": "edges/s",
                "h2d_bytes_per_step": B * C * N * 4, "d2h_bytes_per_step": B * C * N * 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": 4 * args.steps,   # pack weights, fused prologue + node GEMM, tensor-core selection + consumer, exact completion
        "clocks": clk,
        # What binds the dominant kernel: the tcgen05 pre-filter and the CUDA-core top-k bookkeeping that drains its
        # accumulators (tensor pipe + ALU issue).  `frac` is against the measured bf16 tensor peak; the HBM fraction
        # the metric asks for is kept as a secondary block - the kernel is nowhere near HBM bound.
        "roofline": {"bound": "tensor", "co_bound": "alu (top-k filter / list maintenance next to the tensor pipe)",
                     "kernel": "knn_tc4_kernel<28> (four query tiles per CTA: producer warps (TMA ring + tcgen05 "
                               "bf16 (hi,mid) pre-filter) + 16 filter warps with sorting-network list merges, set "
                               "membership by interval arithmetic with exact fp32 chains in the ambiguous band, "
                               "certificate, fused EdgeConv gather/max)",
                     "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s", "frac": achieved / tensor_peak,
                     "flop_per_launch": tensor_flop, "traffic": traffic,
                     "traffic_source": "profiles/traffic.json (ncu --set full dram__bytes_read.sum + dram__bytes_write.sum of "
                                       "one launch; not re-measured in this run)",
                     "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops, burst)", "kernel_ms": kernel_ms,
                     "kernel_share_of_step": kernel_ms / (ms / args.steps),
                     "hbm": {"achieved": hbm_achieved, "peak": peak, "unit": "GB/s", "frac": hbm_achieved / peak,
                             "peak_source": peak_src,
                             "note": "algorithmic bytes = 25.6 B/edge x 1,310,720 edges (read x once, write y once)"}},
    }
    if sustained is not None:
        out["sustained"] = sustained
    if extra is not None:
        out["extra"] = extra
    # ---- baselines on this box (N = 1 only): reference GPU-eager path, reference CPU path ---------------------------
    if world == 1:
        try:
            out["gpu_reference"] = gpu_reference_block(dev, min(args.steps, 10), 2)
            out["gpu_reference"]["speedup_resident"] = out["value"] / out["gpu_reference"]["value"]
        except Exception as exc:
            out["gpu_reference"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
        run = oracle_layer(len(os.sched_getaffinity(0)))
        xc = cpu_sample()
        threads, _ = best_cpu_threads(run, xc, thread_candidates(), args.cpu_seconds * 0.5)
        reps, t0 = 0, time.perf_counter()
        while reps < 3 or (time.perf_counter() - t0 < args.cpu_seconds * 0.5 and reps < 50):
            run(xc)
            reps += 1
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": xc.shape[0] * N * K_NEIGH * reps / dt, "unit": "edges/s", "cores": threads,
                               "kind": "port",
                               "sample": "oracle port of the reference layer on %d of the %d clouds, %d repeats, %.1f s, "
                                         "%d threads = fastest of %s (%d hardware threads available)"
                                         % (xc.shape[0], B, reps, dt, threads, thread_candidates(),
                                            len(os.sched_getaffinity(0)))}
    if last_step is not None:
        dump_outputs(args.dump_outputs, last_step)
    json_out.write(json.dumps(out) + "\n")
    json_out.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_native(a)
