"""TEST INFRASTRUCTURE ONLY -- loads the UNMODIFIED reference modules from /root/reference, or, where that does not
exist (the GPU box), from the byte-for-byte copies `oracle/build_ref.py` placed under oracle/_ref/ (git-ignored).

The reference hot path (`node classification/difformer.py:6-7`,
`physical particle/difformer-v2.py:5-6`) imports two third-party packages that are not
installable in this image (no wheel, no network):

  * torch_sparse 0.6.10  (`node classification/requirements.txt:10`): `SparseTensor(row, col,
    value, sparse_sizes)` + `matmul(adj, x)` (sum-reduce SpMM, duplicates kept and summed)
  * torch_geometric 1.7.2 (`requirements.txt:8`): `utils.degree(index, num_nodes)` =
    occurrence count as float

This file injects minimal stand-ins for exactly those three names (documented semantics of the
pinned versions) so the reference files import *unmodified*.  It is used by
`oracle/make_golden.py` (fixture generation: the tests pin the restatement in
`oracle/difformer_oracle.py` against those recorded reference outputs) and by `bench.py`'s CPU-baseline leg
(the reference's own `full_attention_conv` timed on the host cores).  The product path never
imports it.
"""
import importlib.util
import os
import sys
import types

import torch

_VENDORED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def _pick_root() -> str:
    env = os.environ.get("DIFFORMER_REFERENCE_ROOT")
    for root in ([env] if env else []) + ["/root/reference", _VENDORED]:
        if os.path.isfile(os.path.join(root, "node classification", "difformer.py")):
            return root
    return "/root/reference"


REFERENCE_ROOT = _pick_root()


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "node classification", "difformer.py"))


class _SparseTensor:
    """torch_sparse.SparseTensor stand-in: COO triplets, duplicates preserved."""

    def __init__(self, row=None, col=None, value=None, sparse_sizes=None):
        self.row, self.col, self.value, self.sparse_sizes = row, col, value, sparse_sizes


def _matmul(adj, x):
    """torch_sparse.matmul(adj, x, reduce='sum'): out[adj.row] += adj.value * x[adj.col]."""
    out = torch.zeros((adj.sparse_sizes[0],) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    val = adj.value.to(x.dtype)
    out.index_add_(0, adj.row, val.reshape(-1, *([1] * (x.dim() - 1))) * x[adj.col])
    return out


def _degree(index, num_nodes=None, dtype=None):
    """torch_geometric.utils.degree: float occurrence count of each node id in `index`."""
    n = int(index.max()) + 1 if num_nodes is None else num_nodes
    out = torch.zeros(n, dtype=dtype or torch.float, device=index.device)
    return out.scatter_add_(0, index, torch.ones(index.numel(), dtype=out.dtype, device=index.device))


def install_shims():
    if "torch_sparse" not in sys.modules:
        m = types.ModuleType("torch_sparse")
        m.SparseTensor, m.matmul = _SparseTensor, _matmul
        sys.modules["torch_sparse"] = m
    if "torch_geometric" not in sys.modules:
        pkg = types.ModuleType("torch_geometric")
        utils = types.ModuleType("torch_geometric.utils")
        utils.degree = _degree
        pkg.utils = utils
        sys.modules["torch_geometric"] = pkg
        sys.modules["torch_geometric.utils"] = utils


def _load(path, name):
    install_shims()
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


_cache = {}


def load_reference_v1():
    """`node classification/difformer.py` (full_attention_conv, gcn_conv, DIFFormerConv, DIFFormer)."""
    if "v1" not in _cache:
        _cache["v1"] = _load(os.path.join(REFERENCE_ROOT, "node classification", "difformer.py"),
                             "_reference_difformer_v1")
    return _cache["v1"]


def load_reference_v2():
    """`physical particle/difformer-v2.py` (TransConv, DIFFormer_v2)."""
    if "v2" not in _cache:
        _cache["v2"] = _load(os.path.join(REFERENCE_ROOT, "physical particle", "difformer-v2.py"),
                             "_reference_difformer_v2")
    return _cache["v2"]
