"""GPU tests of the sharded aggregation path: shard-vs-unsharded equality of GCNConv forward and
backward.  The 1-rank case runs on any GPU box; the 2-rank NCCL case needs two GPUs and is
skipped otherwise (the host logic of the 2-rank path is covered on CPU by test_dist_gloo.py)."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _graph(n_total, n_edges, world, seed=7):
    g = torch.Generator().manual_seed(seed)
    n_local = n_total // world
    dst = (torch.rand(n_edges, generator=g) ** 3 * (n_total - 1)).long()
    local = (dst // n_local) * n_local + torch.randint(0, n_local, (n_edges, ), generator=g)
    anywhere = torch.randint(0, n_total, (n_edges, ), generator=g)
    src = torch.where(torch.rand(n_edges, generator=g) < 0.8, local, anywhere)
    x = torch.randn(n_total, 64, generator=g)
    gout = torch.randn(n_total, 128, generator=g)
    w = torch.randn(128, 64, generator=g) / 8
    b = torch.randn(128, generator=g) * 0.1
    return torch.stack([src, dst]), x, gout, w, b


def _run_rank(rank, world, port, n_total, n_edges, q, mode="nccl"):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl" if world > 1 else "gloo", rank=rank, world_size=world)
    try:
        from pytorch_geometric_b200 import dist as pd
        from pytorch_geometric_b200.nn import GCNConv
        ei, x, gout, w, b = _graph(n_total, n_edges, world)
        n_local = n_total // world
        lo = rank * n_local
        conv = GCNConv(64, 128).to(dev)
        with torch.no_grad():
            conv.lin.weight.copy_(w)
            conv.bias.copy_(b)
        # unsharded result on this GPU (the single-process engine, itself parity-checked vs the oracle)
        xg = x.to(dev).requires_grad_()
        ref = conv(xg, ei.to(dev))
        ref.backward(gout.to(dev))
        ref_gx, ref_gw = xg.grad.clone(), conv.lin.weight.grad.clone()
        conv.lin.weight.grad = None
        conv.bias.grad = None
        # sharded
        mine = (ei[1] >= lo) & (ei[1] < lo + n_local)
        xl = x[lo:lo + n_local].to(dev).requires_grad_()
        if mode == "p2p_rgcn":
            # config 5's layer sharded over the ranks: per-relation mean gathered over NVLink, local K = (R+1) F product
            from pytorch_geometric_b200 import dist_p2p
            from pytorch_geometric_b200.graph import cached_graph
            from pytorch_geometric_b200.nn import conv as C
            g = torch.Generator().manual_seed(21)
            R, F = 3, 128
            et = torch.randint(0, R, (ei.size(1), ), generator=g)
            xr = torch.randn(n_total, F, generator=g)
            Wr = (torch.randn(R, F, F, generator=g) / 11).to(dev).requires_grad_()
            root = (torch.randn(F, F, generator=g) / 11).to(dev).requires_grad_()
            bb = (torch.randn(F, generator=g) * 0.1).to(dev).requires_grad_()
            gr = torch.randn(n_total, F, generator=g)
            xg = xr.to(dev).requires_grad_()
            graph = cached_graph(ei.to(dev), n_total, n_total * R, edge_type=et.to(dev), num_relations=R)
            ref = C.rgcn_conv(xg, graph, Wr, root, bb, "mean")
            ref.backward(gr.to(dev))
            ref_gx, ref_gw, ref_groot = xg.grad.clone(), Wr.grad.clone(), root.grad.clone()
            Wr.grad = root.grad = bb.grad = None
            shard = dist_p2p.PeerShardedRelGraph.build(ei[:, mine].to(dev), et[mine].to(dev), R, lo, n_local, n_total, F)
            xl2 = xr[lo:lo + n_local].to(dev).requires_grad_()
            for _ in range(2):
                xl2.grad = None
                Wr.grad = root.grad = bb.grad = None
                out = dist_p2p.peer_sharded_rgcn_conv(Wr, root, bb, xl2, shard)
                out.backward(gr[lo:lo + n_local].to(dev))
            gw2, gr2 = Wr.grad.clone(), root.grad.clone()
            dist.all_reduce(gw2)
            dist.all_reduce(gr2)
            torch.testing.assert_close(out, ref[lo:lo + n_local], rtol=1e-4, atol=1e-4)
            torch.testing.assert_close(xl2.grad, ref_gx[lo:lo + n_local], rtol=1e-4, atol=1e-4)
            torch.testing.assert_close(gw2, ref_gw, rtol=1e-3, atol=1e-3)
            torch.testing.assert_close(gr2, ref_groot, rtol=1e-3, atol=1e-3)
            q.put((rank, "ok"))
            return
        if mode == "p2p_stack":
            # two stacked layers SHARING one shard (one symmetric x W^T buffer), forward-only: the second layer's
            # dense transform overwrites the buffer the first layer's gather read -- legal only because of the
            # barrier after the forward gather (no backward with its barriers runs in between)
            from pytorch_geometric_b200 import dist_p2p
            conv2 = GCNConv(128, 128).to(dev)
            with torch.no_grad():
                conv2.lin.weight.copy_(torch.randn(128, 128, generator=torch.Generator().manual_seed(5)) / 11)
                conv2.bias.copy_(b)
                ref2 = conv2(conv(x.to(dev), ei.to(dev)).relu(), ei.to(dev))
                shard = dist_p2p.PeerShardedGCNGraph.build(ei[:, mine].to(dev), lo, n_local, n_total, 128)
                for _ in range(4):
                    h = dist_p2p.peer_sharded_gcn_conv(conv, xl.detach(), shard).relu()
                    out2 = dist_p2p.peer_sharded_gcn_conv(conv2, h, shard)
                    torch.testing.assert_close(out2, ref2[lo:lo + n_local], rtol=1e-4, atol=1e-4)
            q.put((rank, "ok"))
            return
        if mode == "p2p":
            from pytorch_geometric_b200 import dist_p2p
            shard = dist_p2p.PeerShardedGCNGraph.build(ei[:, mine].to(dev), lo, n_local, n_total, 128)
            for _ in range(2):          # run twice: the second pass exercises the reuse barriers
                xl.grad = None
                conv.lin.weight.grad = None
                conv.bias.grad = None
                out = dist_p2p.peer_sharded_gcn_conv(conv, xl, shard)
                out.backward(gout[lo:lo + n_local].to(dev))
        else:
            shard = pd.ShardedGCNGraph.build(ei[:, mine].to(dev), lo, n_local, n_total)
            out = pd.sharded_gcn_conv(conv, xl, shard)
            out.backward(gout[lo:lo + n_local].to(dev))
        gw = conv.lin.weight.grad.clone()
        if world > 1:
            dist.all_reduce(gw)
        torch.testing.assert_close(out, ref[lo:lo + n_local], rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(xl.grad, ref_gx[lo:lo + n_local], rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(gw, ref_gw, rtol=1e-3, atol=1e-3)
        q.put((rank, "ok"))
    except Exception as exc:
        import traceback
        q.put((rank, "FAIL: " + "".join(traceback.format_exception(exc))))
    finally:
        dist.destroy_process_group()


def _launch(world, mode="nccl"):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_run_rank, args=(r, world, port, 20000, 300000, q, mode)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    for rank, msg in results:
        assert msg == "ok", f"rank {rank}: {msg}"


def test_sharded_gcn_conv_single_rank_equals_unsharded():
    _launch(1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_gcn_conv_two_ranks_nccl_equals_unsharded():
    _launch(2)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_peer_memory_gcn_conv_two_ranks_equals_unsharded():
    """Halo rows gathered over NVLink peer memory inside the kernel (dist_p2p.py)."""
    _launch(2, "p2p")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_peer_memory_two_stacked_layers_share_one_shard_forward_only():
    _launch(2, "p2p_stack")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_peer_memory_rgcn_conv_two_ranks_equals_unsharded():
    """BASELINE config 5 (RGCNConv, 2 x B200): the reduce-agnostic peer-sharded aggregate under the relational layer."""
    _launch(2, "p2p_rgcn")
