"""GPU tests of the reference-side binding: the UNMODIFIED reference package (oracle/_ref, fixture `tg`) running on
cuda with `pytorch_geometric_b200.plugin.install()`, compared with the same reference objects on the CPU (no plug-in
involved there: CPU tensors fall through).

  * the reference's own extension-ABI tests, re-run through the shims: test/utils/test_scatter.py:27-54
    (`torch_scatter.scatter` vs `scatter`) and test/test_edge_index.py:880-929 (`_torch_sparse_spmm` vs `_scatter_spmm`,
    forward + both gradients, all reductions, both transposes);
  * unmodified reference layers (GraphConv / GCNConv / SAGEConv / GINConv) on plain tensors and on sorted `EdgeIndex`
    inputs reach `csr_reduce_kernel` (asserted through the engine's per-op launch profile), never the atomic COO kernel;
  * the subclass layers (`layers=True`) match the reference layers forward and backward, and fall through with hooks;
  * `(out, arg)` operators, the lazy gather's materialisation for messages the fused kernel cannot express.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from pytorch_geometric_b200 import ops  # noqa: E402

DEV = "cuda"


@pytest.fixture
def plugin(tg):
    from pytorch_geometric_b200 import plugin as P
    yield P
    P.uninstall()


def _graph(n=300, e=4000, seed=0, f=32):
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(0, n, (e, ), generator=g)
    dst = (torch.rand(e, generator=g) ** 2 * (n - 1)).long()
    return torch.randn(n, f, generator=g), torch.stack([src, dst])


class _Profile:
    def __enter__(self):
        ops.PROFILE.reset(enabled=True)
        return self

    def __exit__(self, *a):
        self.calls = {k: v["calls"] for k, v in ops.PROFILE.summary().items()}
        ops.PROFILE.reset(enabled=False)
        return False


def _close(a, b, tol=2e-5, what=""):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    err = (a - b).abs().max().item()
    assert err <= tol * max(b.abs().max().item(), 1e-3), f"{what}: max err {err:.3e} vs scale {b.abs().max().item():.3e}"


# ------------------------------------------------------------------------------------------------ the reference's ABI tests
@pytest.mark.parametrize("reduce", ["sum", "add", "mean", "min", "max"])
def test_reference_test_scatter_through_the_torch_scatter_shim(tg, plugin, reduce):
    """test/utils/test_scatter.py:27-54 with `torch_scatter` = the shim module."""
    from torch_geometric.utils import scatter
    from pytorch_geometric_b200.plugin import shims
    torch_scatter = shims.torch_scatter_module()
    torch.manual_seed(1)
    src = torch.randn(100, 16, device=DEV)
    index = torch.randint(0, 8, (100, ), device=DEV)
    out1 = scatter(src, index, dim=0, reduce=reduce)                   # the reference's ATen path on cuda
    out2 = torch_scatter.scatter(src, index, dim=0, reduce=reduce)
    assert out2.device == src.device and torch.allclose(out1, out2, atol=1e-6)
    src = torch.randn(8, 100, 16, device=DEV)
    out1 = scatter(src, index, dim=1, reduce=reduce)
    out2 = torch_scatter.scatter(src, index, dim=1, reduce=reduce)
    assert torch.allclose(out1, out2, atol=1e-6)


@pytest.mark.parametrize("reduce", ["sum", "mean", "min", "max"])
@pytest.mark.parametrize("transpose", [False, True])
@pytest.mark.parametrize("is_undirected", [False, True])
def test_reference_test_torch_sparse_spmm_through_the_registered_ops(tg, plugin, reduce, transpose, is_undirected):
    """test/test_edge_index.py:880-929: the reference's own `_torch_sparse_spmm` (it calls torch.ops.torch_sparse.*)
    against its `_scatter_spmm`, forward and both gradients."""
    import torch_geometric.typing as T
    from torch_geometric import EdgeIndex
    from torch_geometric.edge_index import _scatter_spmm, _torch_sparse_spmm
    from pytorch_geometric_b200.plugin import shims
    assert shims.register_torch_sparse_ops()
    old = T.WITH_TORCH_SPARSE
    T.WITH_TORCH_SPARSE = True                                          # `assert WITH_TORCH_SPARSE` at edge_index.py:1777
    try:
        if is_undirected:
            adj = EdgeIndex([[0, 1, 1, 2], [1, 0, 2, 1]], device=DEV, is_undirected=True)
        else:
            adj = EdgeIndex([[0, 1, 1, 2], [2, 0, 1, 2]], device=DEV)
        adj = adj.sort_by("col" if transpose else "row").values
        torch.manual_seed(3)
        x = torch.randn(3, 1, device=DEV)
        assert _torch_sparse_spmm(adj, x, None, reduce, transpose).allclose(_scatter_spmm(adj, x, None, reduce, transpose), atol=1e-6)
        value = torch.rand(adj.size(1), device=DEV)
        assert _torch_sparse_spmm(adj, x, value, reduce, transpose).allclose(_scatter_spmm(adj, x, value, reduce, transpose), atol=1e-6)
        x1 = torch.randn(3, 1, device=DEV, requires_grad=True)
        x2 = x1.detach().requires_grad_()
        grad = torch.randn_like(x1)
        _torch_sparse_spmm(adj, x1, None, reduce, transpose).backward(grad)
        _scatter_spmm(adj, x2, None, reduce, transpose).backward(grad)
        assert x1.grad.allclose(x2.grad, atol=1e-6)
        v1 = torch.rand(adj.size(1), device=DEV, requires_grad=True)
        v2 = v1.detach().requires_grad_()
        _torch_sparse_spmm(adj, x, v1, reduce, transpose).backward(grad)
        _scatter_spmm(adj, x, v2, reduce, transpose).backward(grad)
        assert v1.grad.allclose(v2.grad, atol=1e-6)
    finally:
        T.WITH_TORCH_SPARSE = old


def test_edge_index_matmul_is_routed_with_its_cached_structure(tg, plugin):
    """EdgeIndex.matmul / `@` on cuda (edge_index.py:1925-1970) -> the CSR kernel on the EdgeIndex's own indptr
    (no re-sort: sort_by_key is never launched), forward + gradients wrt the dense operand and the values."""
    from torch_geometric import EdgeIndex
    x, ei = _graph(200, 3000, 4, 64)
    plugin.install()
    for transpose, order in ((False, "row"), (True, "col")):
        adj_c = EdgeIndex(ei, sparse_size=(200, 200)).sort_by(order).values
        adj_c.fill_cache_()
        adj_g = adj_c.to(DEV)
        adj_g.fill_cache_()
        val = torch.rand(ei.size(1))
        for reduce in ("sum", "mean", "min", "max"):
            xc = x.clone().requires_grad_()
            xg = x.clone().to(DEV).requires_grad_()
            want = adj_c.matmul(xc, input_value=val, reduce=reduce, transpose=transpose)
            with _Profile() as p:
                got = adj_g.matmul(xg, input_value=val.to(DEV), reduce=reduce, transpose=transpose)
            assert p.calls.get("spmm_csr", 0) == 1, p.calls
            _close(got, want, what=f"matmul {reduce} T={transpose}")
            if reduce in ("sum", "mean"):
                gout = torch.randn_like(want)
                want.backward(gout)
                got.backward(gout.to(DEV))
                _close(xg.grad, xc.grad, what=f"matmul grad {reduce}")
    assert "_b200_graphs" in adj_g.__dict__ and adj_g.__dict__["_b200_graphs"][True].perm is None


# ------------------------------------------------------------------------------------------------ unmodified layers
def _run_ref_layer(tg, make, x, ei_cpu, ei_gpu, extra_cpu=(), extra_gpu=()):
    torch.manual_seed(7)
    ref = make()
    gpu = make()
    gpu.load_state_dict(ref.state_dict())
    gpu = gpu.to(DEV)
    xc = x.clone().requires_grad_()
    xg = x.clone().to(DEV).requires_grad_()
    want = ref(xc, ei_cpu, *extra_cpu)
    gout = torch.randn_like(want)
    want.backward(gout)
    with _Profile() as p:
        got = gpu(xg, ei_gpu, *extra_gpu)
        got.backward(gout.to(DEV))
    return ref, gpu, xc, xg, want, got, p.calls


@pytest.mark.parametrize("name,kw", [("GraphConv", {}), ("GraphConv", {"aggr": "mean"}), ("GCNConv", {}), ("SAGEConv", {}),
                                     ("SAGEConv", {"aggr": "max"}), ("GINConv", {})])
@pytest.mark.parametrize("container", ["tensor", "edge_index"])
def test_unmodified_reference_layers_reach_the_csr_kernel(tg, plugin, name, kw, container):
    """No layer swap: the reference's classes, the reference's propagate.  With the plug-in installed the collect step
    is lazy and `aggregate` runs `b200mp_spmm_csr` (csr_reduce_kernel); the atomic COO kernel is not launched."""
    from torch_geometric import EdgeIndex
    x, ei = _graph(300, 4000, 5, 32)
    plugin.install()
    if container == "edge_index":
        ei_c = EdgeIndex(ei, sparse_size=(300, 300)).sort_by("col").values
        ei_g = ei_c.to(DEV)
    else:
        ei_c, ei_g = ei, ei.to(DEV)
    if name == "GINConv":
        make = lambda: tg.nn.GINConv(torch.nn.Sequential(torch.nn.Linear(32, 16), torch.nn.ReLU(), torch.nn.Linear(16, 16)))  # noqa: E731
    else:
        make = lambda: getattr(tg.nn, name)(32, 16, **kw)              # noqa: E731
    ref, gpu, xc, xg, want, got, calls = _run_ref_layer(tg, make, x, ei_c, ei_g)
    assert type(gpu).__module__.startswith("torch_geometric.")           # really the reference's class
    assert calls.get("spmm_csr", 0) >= 1, calls
    _close(got, want, what=name)
    _close(xg.grad, xc.grad, tol=5e-5, what=name + " grad_x")
    for (n, pg), (_, pc) in zip(gpu.named_parameters(), ref.named_parameters()):
        _close(pg.grad, pc.grad, tol=1e-4, what=f"{name} grad {n}")


def test_lazy_gather_materialises_for_messages_it_cannot_fuse(tg, plugin):
    """A layer whose message is not `x_j` / `w * x_j`: the lazy rows are gathered exactly as the reference would."""
    from torch_geometric.nn import MessagePassing

    class Odd(MessagePassing):
        def __init__(self):
            super().__init__(aggr="add")

        def forward(self, x, edge_index):
            return self.propagate(edge_index, x=x)

        def message(self, x_j, x_i):
            return torch.tanh(x_j - x_i) * x_j

    x, ei = _graph(100, 900, 6, 16)
    want = Odd()(x, ei)
    plugin.install()
    got = Odd().to(DEV)(x.to(DEV), ei.to(DEV))
    _close(got, want, what="non-fusable message")


# ------------------------------------------------------------------------------------------------ subclass layers
CASES = [("GCNConv", (32, 16), {}), ("GCNConv", (32, 16), {"normalize": False, "bias": False}),
         ("SAGEConv", (32, 16), {"project": True, "normalize": True}), ("GraphConv", (32, 16), {"aggr": "max"}),
         ("GATConv", (32, 8), {"heads": 4}), ("GATConv", (32, 8), {"heads": 2, "concat": False, "residual": True, "edge_dim": 3}),
         ("GATv2Conv", (32, 8), {"heads": 4}), ("GATv2Conv", (32, 6), {"heads": 3, "share_weights": True, "residual": True}),
         ("GATv2Conv", (32, 8), {"heads": 4, "edge_dim": 3}),
         ("GATv2Conv", (32, 8), {"heads": 2, "edge_dim": 3, "add_self_loops": False, "concat": False, "fill_value": 0.5}),
         ("TransformerConv", (32, 8), {"heads": 4}), ("TransformerConv", (32, 8), {"heads": 2, "concat": False, "beta": True}),
         ("TransformerConv", (32, 8), {"heads": 4, "edge_dim": 3}),
         ("TransformerConv", (32, 16), {"heads": 2, "edge_dim": 3, "concat": False, "beta": True}),
         ("RGCNConv", (32, 16, 3), {}), ("RGCNConv", (32, 16, 3), {"num_bases": 2, "aggr": "sum"}),
         ("RGCNConv", (32, 16, 3), {"num_blocks": 4}), ("FastRGCNConv", (32, 16, 3), {})]


@pytest.mark.parametrize("name,args,kw", CASES)
def test_subclass_layers_match_the_reference_layers(tg, plugin, name, args, kw):
    from pytorch_geometric_b200.plugin import conv as PC
    x, ei = _graph(250, 3500, 8, 32)
    extra_c, extra_g = (), ()
    if "RGCN" in name:
        et = torch.randint(0, 3, (ei.size(1), ), generator=torch.Generator().manual_seed(2))
        extra_c, extra_g = (et, ), (et.to(DEV), )
    if kw.get("edge_dim"):
        ea = torch.randn(ei.size(1), 3, generator=torch.Generator().manual_seed(3))
        extra_c, extra_g = (ea, ), (ea.to(DEV), )
    torch.manual_seed(11)
    ref = getattr(tg.nn, name)(*args, **kw)
    ours = getattr(PC, PC.LAYERS[name])(*args, **kw)
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(DEV)
    xc = x.clone().requires_grad_()
    xg = x.clone().to(DEV).requires_grad_()
    want = ref(xc, ei, *extra_c)
    gout = torch.randn_like(want)
    want.backward(gout)
    n0 = ops.LAUNCHES.count
    got = ours(xg, ei.to(DEV), *extra_g)
    got.backward(gout.to(DEV))
    assert ops.LAUNCHES.count > n0
    _close(got, want, tol=5e-5, what=name)
    _close(xg.grad, xc.grad, tol=2e-4, what=name + " grad_x")
    for (n, pg), (_, pc) in zip(ours.named_parameters(), ref.named_parameters()):
        if pc.grad is not None:
            if n == "lin_key.bias":       # softmax is shift invariant: this gradient is exactly 0 up to rounding noise
                assert pg.grad.abs().max().item() < 1e-4 and pc.grad.abs().max().item() < 1e-4
                continue
            _close(pg.grad, pc.grad, tol=5e-4, what=f"{name} grad {n}")


def test_subclass_layer_with_a_hook_falls_through_to_the_reference_propagate(tg, plugin):
    from pytorch_geometric_b200.plugin import conv as PC
    x, ei = _graph(100, 1000, 9, 32)
    plugin.install()
    conv = PC.B200SAGEConv(32, 16).to(DEV)
    seen = []
    conv.register_aggregate_forward_hook(lambda m, i, o: seen.append(tuple(o.shape)))
    out = conv(x.to(DEV), ei.to(DEV))
    assert seen == [(100, 32)] and out.shape == (100, 16)


# ------------------------------------------------------------------------------------------------ (out, arg) operators
def test_scatter_max_and_spmm_max_return_the_arg():
    from pytorch_geometric_b200.plugin import shims
    ts = shims.torch_scatter_module()
    assert shims.register_torch_sparse_ops()
    g = torch.Generator().manual_seed(5)
    src = torch.randn(500, 7, generator=g)
    index = torch.randint(0, 40, (500, ), generator=g)
    index[index == 13] = 12                                              # group 13 is empty
    for which, fn in (("max", torch.Tensor.argmax), ("min", torch.Tensor.argmin)):
        out, arg = getattr(ts, f"scatter_{which}")(src.to(DEV), index.to(DEV), dim=0, dim_size=40)
        for grp in range(40):
            m = (index == grp).nonzero().view(-1)
            if m.numel() == 0:
                assert (arg[grp] == 500).all() and (out[grp] == 0).all()
                continue
            want = m[fn(src[m], dim=0)]
            assert torch.equal(arg[grp].cpu(), want), (which, grp)
            assert torch.equal(out[grp].cpu(), src[want, torch.arange(7)])
    # CSR form
    order = torch.argsort(index, stable=True)
    rowptr = torch.zeros(41, dtype=torch.long)
    rowptr[1:] = torch.bincount(index, minlength=40).cumsum(0)
    col = torch.randint(0, 60, (500, ), generator=g)
    mat = torch.randn(60, 5, generator=g)
    val = torch.rand(500, generator=g)
    out, arg = torch.ops.torch_sparse.spmm_max(rowptr.to(DEV), col.to(DEV), val.to(DEV), mat.to(DEV))
    for r in range(40):
        b, e = int(rowptr[r]), int(rowptr[r + 1])
        if e == b:
            assert (arg[r] == 500).all()
            continue
        prod = val[b:e, None] * mat[col[b:e]]
        assert torch.equal(arg[r].cpu(), b + prod.argmax(0)) and torch.allclose(out[r].cpu(), prod.max(0).values)
    del order


def test_index_bookkeeping_mirrors_match_the_reference(golden):
    """scatter_argmax / group_argsort / group_cat (utils/_scatter.py:145-300) of the standalone mirror vs the reference's own
    functions run on the CPU (tests/golden/index_bookkeeping.npz; tie-free values: the reference leaves ties to the order
    of a duplicate-index assignment)."""
    from pytorch_geometric_b200 import utils as U
    ref = {k: torch.from_numpy(v) for k, v in golden("index_bookkeeping").items()}
    N, src, index = int(ref["N"]), ref["src"].to(DEV), ref["index"].to(DEV)
    assert torch.equal(U.scatter_argmax(src, index, dim_size=N).cpu(), ref["argmax_dim_size"])
    assert torch.equal(U.scatter_argmax(src, index).cpu(), ref["argmax"])
    for tag, kw in (("plain", {}), ("descending", {"descending": True}), ("consecutive", {"return_consecutive": True}),
                    ("stable", {"stable": True, "num_groups": N})):
        got = U.group_argsort(src, index, **kw)
        assert torch.equal(got.cpu(), ref[f"group_argsort_{tag}"]), kw
    got, gi = U.group_cat([ref["x1"].to(DEV), ref["x2"].to(DEV)], [ref["i1"].to(DEV), ref["i2"].to(DEV)], return_index=True)
    assert torch.equal(got.cpu(), ref["group_cat"]) and torch.equal(gi.cpu(), ref["group_cat_index"])
