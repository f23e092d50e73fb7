"""Generates tests/golden/state_dicts.npz and tests/golden/index_bookkeeping.npz by running the UNMODIFIED reference
(pyg-team/pytorch_geometric v2.9.0, pure Python over ATen) on the CPU:

  state_dicts.npz         the reference layers' state_dict for every case of STATE_DICT_CASES (key "<case>|<name>"):
                          the checkpoints test_cabi_cpu.py checks our layers' keys and shapes against and loads;
  index_bookkeeping.npz   seeded inputs and the reference's scatter_argmax / group_argsort / group_cat results
                          (utils/_scatter.py:145-300) for test_gpu_plugin.py::test_index_bookkeeping_mirrors_match_the_reference.

    python tests/golden/make_golden_api.py <reference checkout>
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, sys.argv[1])
import torch_geometric  # noqa: E402
from torch_geometric.utils._scatter import scatter_argmax  # noqa: E402  (not re-exported by utils/__init__)

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(os.path.dirname(HERE)), os.path.dirname(HERE)]
torch.manual_seed(0)                                                  # STATE_DICT_CASES builds its MLPs on import
from test_cabi_cpu import STATE_DICT_CASES  # noqa: E402

sd = {}
for i, (name, args, kw) in enumerate(STATE_DICT_CASES):
    for k, v in getattr(torch_geometric.nn, name)(*args, **kw).state_dict().items():
        sd[f"{i}|{k}"] = v.detach().numpy()
np.savez_compressed(os.path.join(HERE, "state_dicts.npz"), **sd)

g = torch.Generator().manual_seed(12)
N, E = 70, 900
index = torch.randint(0, N - 5, (E, ), generator=g)
src = torch.randperm(E, generator=g).float() * 0.37 - 100.0          # tie-free values
x1, x2 = torch.randn(40, 3, generator=g), torch.randn(25, 3, generator=g)
i1 = torch.sort(torch.randint(0, 9, (40, ), generator=g))[0]
i2 = torch.sort(torch.randint(0, 9, (25, ), generator=g))[0]
out = {"src": src, "index": index, "x1": x1, "x2": x2, "i1": i1, "i2": i2,
       "argmax_dim_size": scatter_argmax(src, index, dim_size=N), "argmax": scatter_argmax(src, index)}
for tag, kw in (("plain", {}), ("descending", {"descending": True}), ("consecutive", {"return_consecutive": True}),
                ("stable", {"stable": True, "num_groups": N})):
    out[f"group_argsort_{tag}"] = torch_geometric.utils.group_argsort(src, index, **kw)
out["group_cat"], out["group_cat_index"] = torch_geometric.utils.group_cat([x1, x2], [i1, i2], return_index=True)
np.savez_compressed(os.path.join(HERE, "index_bookkeeping.npz"), N=np.int64(N), **{k: v.numpy() for k, v in out.items()})
print("wrote state_dicts.npz and index_bookkeeping.npz")
