#!/usr/bin/env python
"""bench.py -- edges/sec of GCNConv forward+backward on a synthetic power-law graph.

Metric (BASELINE.json): "edges/sec (GCNConv fwd+bwd) at 1/2/4/8 B200; achieved HBM GB/s vs peak".
A *step* is one pass of the hot path: GCNConv(F, F) forward + backward (out.backward(grad)) on the
whole graph, graph structure cached (GCNConv(cached=True) semantics in both arms).
edges/sec = E_input * layers / t (E_input counted before self-loop insertion, SURVEY.md 8(d)).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

N=1 workload: N=10M nodes, E=100M edges, F=256, fp32 (the north-star headline shape; inputs of
10 GB >> 126 MB L2, so no explicit L2 flush is needed).  N>1: weak scaling -- every rank owns a
contiguous node range of the same size with the same number of incoming edges, sources outside the
range are halo rows exchanged with one all_to_all per aggregation pass (pytorch_geometric_b200/dist.py).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True           # the benchmark writes nothing into the source tree (it may be read-only)


# --------------------------------------------------------------------------- helpers
def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.file = None

    def start(self):
        try:
            self.file = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu_index)], stdout=self.file,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.file.flush()
        self.file.seek(0)
        sm, mx, power, reasons = [], [], [], set()
        for line in self.file.read().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.file.name)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(device_index: int):
    """Pins this process to the CPUs of the NUMA node its GPU hangs off, so that pinned host buffers are first-touched
    in node-local memory (at N = 8, eight 10 GB/step H2D streams from one node's DRAM and across the socket
    interconnect halved the end-to-end rate).  Returns the node id or None when the topology cannot be read."""
    try:
        props = torch.cuda.get_device_properties(device_index)
        bdf = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


def synth_graph(num_nodes: int, num_edges: int, seed: int, device, lo: int = 0, total_nodes=None,
                p_local: float = 1.0):
    """Seeded synthetic power-law graph (SURVEY.md 8(d)): destination in-degrees follow a truncated
    power law P(deg = k) ~ k^-2.1 (inverse CDF of the equivalent rank-frequency law, hub ids scattered
    by a random permutation), sources uniform.  Duplicates and self loops are left in.  For sharded runs destinations fall in
    [lo, lo + num_nodes) and a fraction p_local of the sources too; the rest is uniform over all
    `total_nodes` (the halo)."""
    g = torch.Generator(device=device).manual_seed(seed)
    u = torch.rand(num_edges, device=device, generator=g, dtype=torch.float64)
    gamma = 2.1                       # in-degree distribution P(deg = k) ~ k^-gamma
    s = 1.0 / (gamma - 1.0)           # <=> rank-frequency law f(rank) ~ rank^-s (s = 0.909)
    # inverse CDF of the continuous rank law on [1, num_nodes]: F(r) = (r^(1-s) - 1) / (n^(1-s) - 1)
    rank = (1.0 + u * (float(num_nodes) ** (1.0 - s) - 1.0)) ** (1.0 / (1.0 - s))
    rank = (rank.long() - 1).clamp_(0, num_nodes - 1)
    dst = torch.randperm(num_nodes, device=device, generator=g)[rank] + lo   # scatter hubs over the id range
    total = total_nodes if total_nodes is not None else num_nodes
    src_local = torch.randint(0, num_nodes, (num_edges, ), device=device, generator=g) + lo
    if p_local >= 1.0 or total == num_nodes:
        src = src_local
    else:
        src_any = torch.randint(0, total, (num_edges, ), device=device, generator=g)
        pick = torch.rand(num_edges, device=device, generator=g) < p_local
        src = torch.where(pick, src_local, src_any)
    return torch.stack([src, dst])


def traffic_bytes(args):
    """dram bytes per launch of the dominant kernel from the committed ncu capture (profiles/), valid for the
    default workload only."""
    if args.traffic_bytes is not None:
        return args.traffic_bytes
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path) and (args.nodes, args.edges, args.feat) == (10_000_000, 100_000_000, 256):
        with open(path) as f:
            t = json.load(f)
        if "spmm_csr_fwd_bytes" in t:
            return {"fwd": t["spmm_csr_fwd_bytes"], "bwd": t["spmm_csr_bwd_bytes"], "mean": t["spmm_csr_bytes_per_launch"]}
        return t["spmm_csr_bytes_per_launch"]
    return None


def pass_bytes(E_prime: int, N: int, F: int, s: int = 4, b_idx: int = 4, b_w: int = 4) -> int:
    """Algorithmic bytes of one CSR aggregation pass (SURVEY.md 8(d)):
    every edge reads one feature row + its column index + its weight, every row is written once,
    rowptr is read once.  No cache-reuse credit."""
    return E_prime * (F * s + b_idx + b_w) + N * F * s + (N + 1) * b_idx


DUMP_BYTES = 60_000_000                  # --dump-outputs: all arrays together stay below 64 MB


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """`--dump-outputs`: the results the timed path returned in its last step, as <out_dir>/<name>.npy in float32 (float64
    stays float64), so that two builds can be compared output for output on the same seeded inputs.  An array larger than
    its share of DUMP_BYTES is cut to a fixed, seeded sample of its rows: arrays with the same number of rows keep the
    same rows, in ascending order."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        t = t.detach()
        t = t if t.dtype == torch.float64 else t.float()
        if t.numel() * t.element_size() > budget:
            keep = budget // (t[0].numel() * t.element_size())
            rows = torch.randperm(t.size(0), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[rows.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


# --------------------------------------------------------------------------- the CPU reference arm
def workload_config(args, world: int) -> dict:
    """The workload both arms are quoted on (identical dict in the b200 and the reference line)."""
    N, E, F = args.nodes, args.edges, args.feat
    return {"workload": f"GCNConv({F},{F}) fwd+bwd, power-law synthetic graph (in-degree exponent 2.1, uniform sources), "
                        f"N={N} nodes and E={E} edges per GPU, fp32, graph cached (cached=True)",
            "nodes_per_gpu": N, "edges_per_gpu": E, "feat": F, "layers": 1, "n_gpus": world}


def _import_reference():
    """The UNMODIFIED reference package, where build() installed it (oracle/install_ref.sh; git-ignored)."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    if os.path.isdir(os.path.join(ref, "torch_geometric")):
        if ref not in sys.path:
            sys.path.insert(0, ref)
        import torch_geometric
        return torch_geometric
    return None


def _cpu_threads() -> int:
    """Host threads for the CPU arm: the physical cores (half the logical CPUs), also under torchrun -- which
    exports OMP_NUM_THREADS=1 to every rank and would otherwise cut the CPU arm to one thread at N > 1."""
    n = max(1, (os.cpu_count() or 2) // 2)
    torch.set_num_threads(n)
    return torch.get_num_threads()


def _reference_step_fn(args):
    """(step, kind, how): one GCNConv(F, F, cached=True) forward+backward on the bounded CPU sample -- through the
    reference's own GCNConv when oracle/_ref is installed, else through the restated ATen call sequence."""
    N, E, F = args.cpu_nodes, args.cpu_edges, args.feat
    torch.manual_seed(0)
    ei = synth_graph(N, E, 1, "cpu")
    x = torch.randn(N, F, requires_grad=True)
    gout = torch.randn(N, F)
    tg = _import_reference()
    if tg is not None:
        conv = tg.nn.GCNConv(F, F, cached=True)

        def step():
            x.grad = None
            conv.zero_grad(set_to_none=True)
            conv(x, ei).backward(gout)
        return step, "reference", f"torch_geometric {tg.__version__} GCNConv (oracle/_ref, unmodified), default [2,E] tensor path"
    from oracle import ref_aten
    weight = torch.nn.Parameter(torch.randn(F, F) / F ** 0.5)
    bias = torch.nn.Parameter(torch.zeros(F))
    ei2, w2 = ref_aten.gcn_norm(ei, None, N)                          # cached=True: outside the loop

    def step():
        x.grad = weight.grad = bias.grad = None
        ref_aten.gcn_conv_forward(x, ei2, w2, weight, bias).backward(gout)
    return step, "port", "oracle/ref_aten.py (the reference's ATen call sequence; oracle/_ref not installed)"


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path, timed on the host cores on a bounded
    sample of the workload, exactly --warmup W untimed and --steps K timed steps.  Rank 0 only under torchrun."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = _cpu_threads()
    step, kind, how = _reference_step_fn(args)
    N, E, F = args.cpu_nodes, args.cpu_edges, args.feat
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    value = E / dt
    sample = (f"{how}; bounded sample of the workload: N={N}, E={E} (same generator), F={F}, fp32, "
              f"{args.steps} steps, {cores} torch threads of {os.cpu_count()} host CPUs")
    emit({
        "impl": "reference", "metric": "edges/sec (GCNConv fwd+bwd)", "value": value, "unit": "edges/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": "edges/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def cpu_baseline_quick(args):
    """Bounded CPU sample for the `cpu_baseline` object of the main line (rank 0, N=1 only)."""
    cores = _cpu_threads()
    step, kind, how = _reference_step_fn(args)
    N, E, F = args.cpu_nodes, args.cpu_edges, args.feat
    step()
    t0 = time.perf_counter()
    n = 0
    while n < 3 and (n == 0 or time.perf_counter() - t0 < 20):
        step()
        n += 1
    dt = (time.perf_counter() - t0) / n
    return {"value": E / dt, "unit": "edges/s", "cores": cores, "kind": kind,
            "sample": f"{how}; GCNConv({F},{F}) fwd+bwd on N={N}, E={E} (same generator), {n} steps, "
                      f"{cores} torch threads of {os.cpu_count()} host CPUs"}


# --------------------------------------------------------------------------- parity at the benchmarked size
def run_parity(args, conv, fwd, step, ei, x, gout, rank, world, dev):
    """`parity_check` of the JSON line.  (1) The timed step's out / grad_x / grad_W / grad_b on a seeded sample of
    destination and source rows (hubs, rows with 0 / 1 / 2 edges, random rows) against the CPU oracle restricted to
    those rows (oracle/sampled.py), at 1e-5 * sum|terms|.  (2) N > 1: additionally the sharded engine against the
    unsharded engine on a graph small enough for one GPU, through the very same code path the timed loop used."""
    import torch.distributed as dist

    from oracle import sampled
    N = args.nodes
    out = step()
    gw, gb = conv.lin.weight.grad, conv.bias.grad
    res = sampled.gcn_check(ei, rank * N, N, x, conv.lin.weight, conv.bias, gout, out, x.grad, gw, gb,
                            n_rows=args.parity_rows, seed=17, group=dist.group.WORLD if world > 1 else None)
    del out
    if world > 1:
        res["sharded_vs_unsharded"] = shard_vs_unsharded(args, conv, rank, world, dev)
        res["ok"] = bool(res["ok"] and res["sharded_vs_unsharded"]["ok"])
    return res


# Both sides of this comparison are fp32 engine results that differ only in summation order (per-rank partial weight
# gradients + all_reduce vs one split-K GEMM; shard-local vs global edge order), and the difference is measured against
# the row's largest |value|, not against sum|terms| -- so the bound is looser than parity_check's 1e-5 (which is the
# oracle comparison).  Measured: 1.8e-5 at N = 2.
SHARD_TOL = 1e-4


def shard_vs_unsharded(args, conv, rank, world, dev, n_small=100_000, e_small=1_000_000):
    """Every rank builds the WHOLE small graph (all ranks' seeded edge lists), runs the single-GPU engine on it, and
    compares its own rows with what the sharded path (same builder, same kernels, same barriers as the timed loop)
    produces; grad_W / grad_b after the all-reduce."""
    import torch.distributed as dist

    from pytorch_geometric_b200 import utils as U
    F = args.feat
    eis = [synth_graph(n_small, e_small, 1000 + q, dev, lo=q * n_small, total_nodes=world * n_small, p_local=args.p_local)
           for q in range(world)]
    xs = [torch.randn(n_small, F, device=dev, generator=torch.Generator(device=dev).manual_seed(2000 + q)) for q in range(world)]
    gs = [torch.randn(n_small, F, device=dev, generator=torch.Generator(device=dev).manual_seed(3000 + q)) for q in range(world)]
    x_full = torch.cat(xs).requires_grad_()
    graph = U.gcn_norm_graph(torch.cat(eis, dim=1), None, world * n_small)
    conv.zero_grad(set_to_none=True)
    ref = conv(x_full, graph)
    ref.backward(torch.cat(gs))
    ref_gw, ref_gb = conv.lin.weight.grad.clone(), conv.bias.grad.clone()
    lo = rank * n_small
    ref_out, ref_gx = ref.detach()[lo:lo + n_small].clone(), x_full.grad[lo:lo + n_small].clone()
    del ref, x_full, graph
    conv.zero_grad(set_to_none=True)
    xl = xs[rank].clone().requires_grad_()
    if args.dist == "p2p":
        from pytorch_geometric_b200 import dist_p2p
        shard = dist_p2p.PeerShardedGCNGraph.build(eis[rank], lo, n_small, world * n_small, F, dist.group.WORLD)
        shard.gout.copy_(gs[rank])
        for _ in range(2):                                   # twice: the second pass exercises the reuse barriers
            xl.grad = None
            conv.zero_grad(set_to_none=True)
            out = dist_p2p.peer_sharded_gcn_conv(conv, xl, shard)
            out.backward(shard.gout)
    else:
        from pytorch_geometric_b200 import dist as pdist
        shard = pdist.ShardedGCNGraph.build(eis[rank], lo, n_small, world * n_small, dist.group.WORLD)
        out = pdist.sharded_gcn_conv(conv, xl, shard)
        out.backward(gs[rank])
    gw, gb = conv.lin.weight.grad.clone(), conv.bias.grad.clone()
    dist.all_reduce(gw)
    dist.all_reduce(gb)

    def rel(a, b):                                            # relative to the row's magnitude (sum of |terms| proxy)
        scale = b.abs().amax(dim=-1, keepdim=True).clamp(min=1e-20) if b.dim() > 1 else b.abs().max().clamp(min=1e-20)
        return float(((a - b).abs() / scale).max())

    per = {"out": rel(out.detach(), ref_out), "grad_x": rel(xl.grad, ref_gx), "grad_W": rel(gw, ref_gw), "grad_b": rel(gb, ref_gb)}
    t = torch.tensor([max(per.values())], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    conv.zero_grad(set_to_none=True)
    return {"nodes": world * n_small, "edges": world * e_small, "p_local": args.p_local, "path": args.dist,
            "max_rel": float(t.item()), "tol": SHARD_TOL, "ok": bool(t.item() <= SHARD_TOL), "per_quantity_rank0": per}


# --------------------------------------------------------------------------- the B200 arm
def run_b200(args):
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import pytorch_geometric_b200 as pgb
    from pytorch_geometric_b200 import ops
    from pytorch_geometric_b200 import utils as U
    from pytorch_geometric_b200.nn import GCNConv

    N, E, F = args.nodes, args.edges, args.feat
    ops.set_option("spmm_impl", args.spmm_impl)
    ops.set_option("spmm_tune", args.spmm_tune)
    from pytorch_geometric_b200 import dense
    dense.set_backend(args.dense)
    if args.gemm_bk:
        ops.set_option("gemm_bk", args.gemm_bk)
    if args.gemm_mode >= 0:
        ops.set_option("gemm_mode", args.gemm_mode)
    if args.gemm_prefetch >= 0:
        ops.set_option("gemm_prefetch", args.gemm_prefetch)
    if args.gemm_bsplit >= 0:
        dense.set_b_split(bool(args.gemm_bsplit))
    torch.manual_seed(1234)                  # the SAME layer parameters on every rank (what DDP's broadcast guarantees)
    conv = GCNConv(F, F, cached=True).to(dev)
    with torch.no_grad():
        conv.bias.normal_(0, 0.1)
    if world == 1:
        ei = synth_graph(N, E, 1, dev)
        graph = U.gcn_norm_graph(ei, None, N)
        graph.build_transpose()
        halo = None
        E_prime = graph.num_edges
        fwd = lambda xx: conv(xx, graph)                                     # noqa: E731
    else:
        ei = synth_graph(N, E, 1 + rank, dev, lo=rank * N, total_nodes=world * N, p_local=args.p_local)
        shard = None
        if args.dist == "p2p":
            # halo exchange fused into the gather kernel over NVLink peer memory (dist_p2p.py)
            try:
                from pytorch_geometric_b200 import dist_p2p
                shard = dist_p2p.PeerShardedGCNGraph.build(ei, rank * N, N, world * N, F, dist.group.WORLD)
                fwd = lambda xx: dist_p2p.peer_sharded_gcn_conv(conv, xx, shard)    # noqa: E731
            except Exception as exc:                                  # symmetric memory unavailable on this box
                print(f"[bench] symmetric-memory path unavailable ({exc!r}); using the NCCL all_to_all path", file=sys.stderr)
                args.dist = "nccl"
                shard = None
        if shard is None:
            from pytorch_geometric_b200 import dist as pdist
            shard = pdist.ShardedGCNGraph.build(ei, rank * N, N, world * N, dist.group.WORLD)
            fwd = lambda xx: pdist.sharded_gcn_conv(conv, xx, shard)             # noqa: E731
        E_prime = shard.num_edges
        graph = shard.graph
        # edges whose source row lives on another GPU: every one reads a full feature row over NVLink per pass
        remote = ((ei[0] < rank * N) | (ei[0] >= (rank + 1) * N)).sum().to(torch.float64)
        dist.all_reduce(remote, op=dist.ReduceOp.MAX)
        remote_edges = int(remote.item())
    torch.cuda.synchronize()

    gen = torch.Generator(device=dev).manual_seed(4321 + rank)
    x = torch.randn(N, F, device=dev, generator=gen).requires_grad_()
    if world > 1 and args.dist == "p2p":
        gout = shard.gout.normal_(generator=gen)                      # upstream gradient produced in the symmetric buffer
    else:
        gout = torch.randn(N, F, device=dev, generator=gen)

    def step():
        x.grad = None
        conv.lin.weight.grad = None
        conv.bias.grad = None
        out = fwd(x)
        out.backward(gout)
        if world > 1:                       # data-parallel weight gradients, as DDP would do
            dist.all_reduce(conv.lin.weight.grad)
            dist.all_reduce(conv.bias.grad)
        return out

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ops.PROFILE.reset(enabled=True)
    launches0 = ops.LAUNCHES.count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    ev0.record()
    out = None
    for _ in range(args.steps):
        out = None                          # released before the next step allocates, as if it were not kept
        out = step()
    ev1.record()
    sync_all()
    ms = ev0.elapsed_time(ev1)
    launches = ops.LAUNCHES.count - launches0
    kern = ops.PROFILE.summary()                                              # per-kernel CUDA-event times
    ops.PROFILE.reset(enabled=False)
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    value = world * E / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"out": out, "grad_x": x.grad, "grad_weight": conv.lin.weight.grad,
                                         "grad_bias": conv.bias.grad})
    del out

    # ---- end to end through the public API with HOST buffers (N=1 path; per rank for N>1)
    e2e = None
    numa_node = None
    if not args.no_e2e:
        numa_node = bind_to_gpu_numa_node(local_rank)                         # before the pinned buffer is first touched
        x_host = torch.empty(N, F, dtype=torch.float32, pin_memory=True)
        x_host.normal_()
        # Input prefetch, as a training loop with a pinned-memory loader does it: two device buffers,
        # the H2D copy of step i+1 runs on a copy stream while step i computes.  Every step still
        # pays its own full H2D copy and its own D2H read inside the timed region.
        x_bufs = [torch.empty(N, F, device=dev) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=dev)
        main_stream = torch.cuda.current_stream(dev)
        gw_host = torch.empty(F, F, dtype=torch.float32, pin_memory=True)
        gb_host = torch.empty(F, dtype=torch.float32, pin_memory=True)
        loss_host = torch.empty(1, dtype=torch.float32, pin_memory=True)
        for ev in freed:
            ev.record(main_stream)

        def prefetch(i):
            b = i & 1
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[b])                              # buffer no longer read by step i-2
                x_bufs[b].copy_(x_host, non_blocking=True)                    # H2D of step i's input
                ready[b].record(copy_stream)

        def e2e_step(i):
            b = i & 1
            prefetch(i + 1)
            main_stream.wait_event(ready[b])
            xin = x_bufs[b].detach().requires_grad_()
            conv.lin.weight.grad = None
            conv.bias.grad = None
            out = fwd(xin)
            loss = (out * gout).sum()                                         # the step's scalar result
            out.backward(gout)
            if world > 1:
                dist.all_reduce(conv.lin.weight.grad)
                dist.all_reduce(conv.bias.grad)
            gw_host.copy_(conv.lin.weight.grad, non_blocking=True)            # D2H of the step's results
            gb_host.copy_(conv.bias.grad, non_blocking=True)
            loss_host.copy_(loss.detach().view(1), non_blocking=True)
            freed[b].record(main_stream)

        prefetch(0)
        for i in range(2):
            e2e_step(i)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_e2e = max(3, min(args.steps, 10))
        e0.record()
        for i in range(2, 2 + n_e2e):
            e2e_step(i)
        e1.record()
        sync_all()
        ems = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ems], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
        e2e = {"value": world * E / (ems / n_e2e * 1e-3), "unit": "edges/s",
               "h2d_bytes_per_step": world * N * F * 4, "d2h_bytes_per_step": world * (F * F + F + 1) * 4,
               "ms_per_step": ems / n_e2e, "steps": n_e2e,
               "host_link_gbs_per_gpu": N * F * 4 / (ems / n_e2e * 1e-3) / 1e9, "numa_node_of_pinned_buffer": numa_node,
               "what": "pinned-host x -> H2D (prefetched one step ahead on a copy stream, double-buffered) -> "
                       "GCNConv fwd+bwd -> D2H of grad_W, grad_b and the loss scalar, every step; "
                       "bound by the 10.24 GB/step host link"}
        del x_host, x_bufs

    # ---- parity at the benchmarked size: one more step, then a seeded row sample against the CPU oracle
    parity = None
    if not args.no_parity:
        parity = run_parity(args, conv, fwd, step, ei, x, gout, rank, world, dev)
    del ei

    if rank == 0:
        peak, peak_src = measured_peaks()
        bytes_pass = pass_bytes(E_prime, N, F)
        agg = kern.get("spmm_csr", {"ms_total": 0.0, "calls": 0, "ms_each": []})
        avg_ms = agg["ms_total"] / max(agg["calls"], 1)
        achieved = bytes_pass / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
        traffic = traffic_bytes(args) if world == 1 else None
        # launches alternate forward (destination-sorted CSR) / backward (source-sorted CSR) inside a step
        by_pass = {}
        each = agg.get("ms_each", [])
        for name, sl in (("fwd", each[0::2]), ("bwd", each[1::2])):
            if sl:
                m_ = sum(sl) / len(sl)
                a_ = bytes_pass / (m_ * 1e-3) / 1e9
                t_ = traffic.get(name) if isinstance(traffic, dict) else None
                by_pass[name] = {"avg_launch_ms": m_, "achieved": a_, "frac": a_ / peak, "traffic": t_,
                                 "frac_on_traffic": (t_ / (m_ * 1e-3) / 1e9 / peak) if t_ else None}
        roofline = {"bound": "hbm", "kernel": "csr_reduce_kernel (b200mp_spmm_csr), fwd on CSR + bwd on transposed CSR",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": bytes_pass,
                    "avg_launch_ms": avg_ms, "launches_timed": agg["calls"],
                    "share_of_step": agg["ms_total"] / ms if ms > 0 else None,
                    "traffic": (traffic.get("mean") if isinstance(traffic, dict) else traffic),
                    "traffic_source": ("profiles/traffic.json (ncu --set full capture of this command at this shape, "
                                       "dram__bytes_read.sum + dram__bytes_write.sum per launch)" if traffic else
                                       "null: no committed ncu capture for this shape / rank count"),
                    "by_pass": by_pass, "frac_of_nominal_8TBs": achieved / 8000.0}
        cpu = None
        if world == 1 and not args.no_cpu:
            cpu = cpu_baseline_quick(args)
        line = {
            "metric": "edges/sec (GCNConv fwd+bwd)", "value": value, "unit": "edges/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": workload_config(args, world),
            "engine": {"edges_with_self_loops": E_prime, "index_dtype": "int32",
                       "l2_policy": "inputs (x, grad, CSR > 10 GB) are far larger than the 126 MB L2; no explicit flush",
                       "parallelism": "single GPU" if world == 1 else (
                           f"node-range sharding x{world}, p_local={args.p_local}, " +
                           ("halo rows gathered over NVLink peer memory inside the kernel (symmetric memory)"
                            if args.dist == "p2p" else "halo all_to_all (NCCL) overlapped with the local sweep")),
                       "gemm": ("hand-written tcgen05 3xTF32, A operand in TMEM (fp32-accurate, csrc/gemm_tf32x3.cu + gemm_tf32x3_ts.cuh)" if args.dense == "tf32x3"
                                else "torch.nn.functional.linear (cuBLAS fp32, allow_tf32=False)"),
                       "halo": (None if world == 1 else {
                           "remote_edges_per_gpu_max": remote_edges, "remote_edge_fraction": remote_edges / max(E_prime, 1),
                           "nvlink_read_bytes_per_pass_per_gpu": remote_edges * F * 4,
                           "nvlink_gbs_per_gpu_in_gather": (remote_edges * F * 4 / (avg_ms * 1e-3) / 1e9) if avg_ms > 0 else None,
                           "note": "every remote edge reads one full feature row from the owner's HBM over NVLink inside "
                                   "csr_reduce_kernel (no dedup: sources are uniform, repeats are rare); 900 GB/s per direction per GPU"}),
                       "long_rows": graph.plan.n_long, "chunks": graph.plan.n_chunks,
                       "spmm_impl": {0: "default (register-staged lane-group kernel, csrc/csr_reduce.cuh)", 1: "lane-group kernel",
                                     2: "persistent TMA-fed variant (csrc/csr_tma.cuh)"}[args.spmm_impl]},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "parity_check": parity, "gpu_launches": launches,
            "kernels": {k: {"ms_total": v["ms_total"], "calls": v["calls"]} for k, v in kern.items()}, "clocks": clocks,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """Exactly ONE JSON line on the real stdout (libraries such as NCCL print banners to fd 1,
    so fd 1 is pointed at stderr for the whole run and the result goes to the saved descriptor)."""
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nodes", type=int, default=10_000_000, help="nodes per GPU")
    ap.add_argument("--edges", type=int, default=100_000_000, help="edges per GPU")
    ap.add_argument("--feat", type=int, default=256)
    ap.add_argument("--dist", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: halo rows gathered over NVLink peer memory inside the kernel, or NCCL all_to_all")
    ap.add_argument("--p-local", type=float, default=0.95, help="fraction of sources inside the owner's range (N>1)")
    ap.add_argument("--cpu-nodes", type=int, default=250_000)
    ap.add_argument("--cpu-edges", type=int, default=2_500_000)
    ap.add_argument("--spmm-impl", type=int, default=0, help="0 auto, 1 lane-group kernel, 2 TMA kernel")
    ap.add_argument("--spmm-tune", type=int, default=0, help="tuning variant of the lane-group kernel (csr_reduce.cuh)")
    ap.add_argument("--dense", default="tf32x3", choices=["tf32x3", "cublas"],
                    help="dense transform: hand-written tcgen05 3xTF32 GEMM (fp32-accurate) or strict-fp32 cuBLAS")
    ap.add_argument("--gemm-bk", type=int, default=0, help="k-block width of the tcgen05 GEMM (16 or 32; 0 = library default)")
    ap.add_argument("--gemm-prefetch", type=int, default=-1, help="TMA L2-prefetch distance of the GEMM in k-blocks")
    ap.add_argument("--gemm-mode", type=int, default=-1, help="0 = SS-mode GEMM, 1 = TS-mode (A in TMEM); -1 = library default")
    ap.add_argument("--gemm-bsplit", type=int, default=-1,
                    help="1 = the GEMM kernel splits W tiles itself (one L2 read of W per tile), 0 = pre-split W_hi / W_lo")
    ap.add_argument("--config", type=int, default=0,
                    help="0 = the headline (GCNConv); 2 / 3 / 5 = the other single-box BASELINE configs (benchmarks/configs.py)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the sampled-row oracle check after the timed loop")
    ap.add_argument("--parity-rows", type=int, default=4096)
    ap.add_argument("--traffic-bytes", type=float, default=None,
                    help="dram bytes per launch of the dominant kernel from the committed ncu capture (profiles/)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (output, gradients of the input and "
                         "of the parameters) as DIR/<name>.npy; at N > 1 rank 0's rows; not with --impl reference")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs records the B200 path; the reference arm has nothing to dump")
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
        if args.config:
            from benchmarks import configs
            configs.run_config(args, sys.modules[__name__])
        else:
            run_b200(args)


if __name__ == "__main__":
    main()
