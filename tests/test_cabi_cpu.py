"""CPU-side checks of the boundary: the C-ABI library loads without a GPU, exports every symbol
include/b200mp.h declares, and the host-side mirror refuses to run anywhere but on CUDA."""
import numpy as np
import pytest
import torch

import pytorch_geometric_b200 as pgb
from pytorch_geometric_b200 import _lib, ops, utils as U
from pytorch_geometric_b200.nn import GCNConv, SumAggregation


def test_library_loads_and_exports_every_declared_symbol():
    lib = pgb.lib()
    syms = pgb.header_symbols()
    assert len(syms) >= 25
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, missing
    assert lib.b200mp_version() == b"0.1.0"
    # every symbol the Python binding declares is in the header, and vice versa
    assert sorted(_lib._SIGS) == syms


def test_no_cpu_fallback():
    x = torch.randn(4, 8)
    idx = torch.tensor([0, 1, 1, 3])
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.scatter_coo(x, idx, 4, "sum")
    with pytest.raises(RuntimeError, match="CUDA"):
        U.scatter(x, idx, 0, 4, "sum")
    with pytest.raises(RuntimeError, match="CUDA"):
        pgb.CSRGraph(idx, idx, 4, 4)
    with pytest.raises(RuntimeError):
        GCNConv(8, 8)(x, torch.stack([idx, idx]))


def test_argument_errors_match_reference_messages():
    x = torch.randn(4, 8)
    idx = torch.tensor([0, 1, 1, 3])
    with pytest.raises(ValueError, match="must be one-dimensional"):      # _scatter.py:37-39
        U.scatter(x, idx.view(2, 2), 0, 4)
    with pytest.raises(ValueError, match="must lay between"):            # _scatter.py:43-45
        U.scatter(x, idx, 3, 4)
    with pytest.raises(ValueError, match="invalid `reduce` argument"):   # _scatter.py:138
        U.scatter(x, idx, 0, 4, "foo")
    with pytest.raises(ValueError, match="invalid dimension"):           # aggr/base.py:105-107
        SumAggregation()(x, idx, dim=4)


def test_state_dict_layout_matches_reference_layers():
    sd = GCNConv(8, 16).state_dict()
    assert set(sd) == {"bias", "lin.weight"} and sd["lin.weight"].shape == (16, 8)
    from pytorch_geometric_b200.nn import RGCNConv, SAGEConv
    assert set(SAGEConv(8, 16).state_dict()) == {"lin_l.weight", "lin_l.bias", "lin_r.weight"}
    sd = RGCNConv(8, 16, 3).state_dict()
    assert sd["weight"].shape == (3, 8, 16) and sd["root"].shape == (8, 16) and sd["bias"].shape == (16, )


def _mlp():
    return torch.nn.Sequential(torch.nn.Linear(8, 16), torch.nn.ReLU(), torch.nn.Linear(16, 16))


# (layer, args, kwargs); tests/golden/state_dicts.npz holds the reference layer's state_dict for each case
# (tests/golden/make_golden_api.py), so a change here needs that file regenerated
STATE_DICT_CASES = [
    ("GCNConv", (8, 16), {}), ("SAGEConv", (8, 16), {}), ("SAGEConv", (8, 16), {"project": True}),
    ("GATConv", (8, 4), {"heads": 3}), ("GATConv", (8, 4), {"heads": 2, "concat": False, "residual": True}),
    ("RGCNConv", (8, 16, 3), {}), ("GINConv", (_mlp(), ), {"train_eps": True}), ("GINConv", (_mlp(), ), {}),
    ("GATConv", (8, 4), {"heads": 2, "edge_dim": 3}), ("GATConv", ((8, 6), 4), {"heads": 2}),
    ("GATv2Conv", (8, 4), {"heads": 3, "edge_dim": 5}),
    ("GATv2Conv", (8, 4), {"heads": 2, "share_weights": True, "residual": True, "concat": False}),
    ("TransformerConv", (8, 4), {"heads": 3, "edge_dim": 5, "beta": True}),
    ("TransformerConv", (8, 4), {"heads": 2, "concat": False, "bias": False}),
    ("GraphConv", (8, 16), {}), ("RGCNConv", (8, 16, 3), {"num_bases": 2}), ("RGCNConv", (8, 16, 3), {"num_blocks": 4}),
    ("FastRGCNConv", (8, 16, 3), {}), ("HeteroLinear", (8, 16, 3), {}), ("HeteroLinear", (8, 16, 3), {"bias": False})]


def test_state_dict_names_and_shapes_equal_the_reference_layers(golden):
    """Checkpoints are interchangeable: same keys AND shapes as the reference's layers, option by option (GIN's eps is [1],
    `edge_dim` adds `lin_edge` / `att_edge`, `share_weights` registers one module under two names, ...)."""
    import pytorch_geometric_b200.nn as ours
    ref = {}
    for key, v in golden("state_dicts").items():
        case, name = key.split("|", 1)
        ref.setdefault(int(case), {})[name] = torch.from_numpy(v)
    assert sorted(ref) == list(range(len(STATE_DICT_CASES)))
    for i, (name, args, kw) in enumerate(STATE_DICT_CASES):
        a = getattr(ours, name)(*args, **kw).state_dict()
        b = ref[i]
        assert {k: tuple(v.shape) for k, v in a.items()} == {k: tuple(v.shape) for k, v in b.items()}, (name, kw)
        getattr(ours, name)(*args, **kw).load_state_dict(b)          # a reference checkpoint loads


def test_fused_and_multi_aggregation_argument_errors_match_reference_messages():
    # nn/aggr/fused.py:87-110 and multi.py:52-70,101-110: validated before anything touches the device
    from pytorch_geometric_b200.nn import FusedAggregation, MultiAggregation, StdAggregation, aggregation_resolver
    with pytest.raises(ValueError, match="should be a list or tuple"):
        FusedAggregation("sum")
    with pytest.raises(ValueError, match="should not be empty"):
        FusedAggregation([])
    with pytest.raises(ValueError, match="not fusable"):
        FusedAggregation(["sum", "softmax"])
    f = FusedAggregation(["sum", aggregation_resolver("std", semi_grad=True), "max"])
    assert f.names == ["sum", "std", "max"] and f.semi_grad and repr(f) == "FusedAggregation()"
    with pytest.raises(ValueError, match="should be a list or tuple"):
        MultiAggregation("sum")
    with pytest.raises(ValueError, match="should not be empty"):
        MultiAggregation([])
    with pytest.raises(ValueError, match="invalid length"):
        MultiAggregation(["sum", "max"], aggrs_kwargs=[{}])
    with pytest.raises(ValueError, match="Multiple aggregations are required"):
        MultiAggregation(["sum"], mode="proj", mode_kwargs=dict(in_channels=4, out_channels=2))
    with pytest.raises(ValueError, match="must have `in_channels` and `out_channels`"):
        MultiAggregation(["sum", "max"], mode="proj")
    m = MultiAggregation(["mean", "min", "max", "std"])
    assert m.get_out_channels(16) == 64 and m.is_fused == [True] * 4
    assert isinstance(m.aggrs[3], StdAggregation)
    assert MultiAggregation(["sum", "softmax"], mode="proj", mode_kwargs=dict(in_channels=4, out_channels=3)).get_out_channels(4) == 3
    # no CPU fallback here either
    with pytest.raises(RuntimeError, match="CUDA"):
        f(torch.randn(4, 8), torch.tensor([0, 1, 1, 3]), dim_size=4)


def test_multi_aggr_wrapper_rejects_unknown_names_without_a_gpu():
    from pytorch_geometric_b200 import functional as Fn
    with pytest.raises(ValueError, match="cannot fuse aggregation 'mul'"):
        Fn.multi_aggregate((torch.zeros(2, dtype=torch.long), torch.zeros(1, dtype=torch.long)), torch.randn(1, 4), ["sum", "mul"])
    with pytest.raises(ValueError, match="duplicate"):
        Fn.multi_aggregate((torch.zeros(2, dtype=torch.long), torch.zeros(1, dtype=torch.long)), torch.randn(1, 4), ["sum", "add"])


def test_prebuilt_library_is_matched_by_content_not_by_file_time():
    """The .so built here travels to the GPU box in a snapshot whose file times carry no meaning: staleness
    is decided by a fingerprint of the sources, so touching a file must not trigger minutes of nvcc there."""
    import os

    from pytorch_geometric_b200 import _build
    _build.build()
    assert not _build.needs_build()
    src = _build.sources()[0]
    st = os.stat(src)
    try:
        os.utime(src)                                     # newer than the .so now
        assert not _build.needs_build()
    finally:
        os.utime(src, (st.st_atime, st.st_mtime))
    with open(_build.STAMP) as fh:
        good = fh.read()
    try:
        with open(_build.STAMP, "w") as fh:
            fh.write("0" * 64 + "\n")
        assert _build.needs_build()                       # a different fingerprint does
    finally:
        with open(_build.STAMP, "w") as fh:
            fh.write(good)
    assert not _build.needs_build()


def test_header_is_plain_c_and_cxx(tmp_path):
    """include/b200mp.h is the boundary: it must compile as C99 and as C++ with nothing but <stdint.h> (no torch types)."""
    import os
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "use_header.c"
    src.write_text('#include "b200mp.h"\nint main(void) { return b200mp_version() == 0; }\n')
    inc = os.path.join(root, "include")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-I", inc, str(src)], check=True)
    subprocess.run(["g++", "-std=c++17", "-Wall", "-Werror", "-fsyntax-only", "-x", "c++", "-I", inc, str(src)], check=True)
    text = open(os.path.join(inc, "b200mp.h")).read()
    assert "#include <torch" not in text and "at::Tensor" not in text and "c10::" not in text
