"""CPU: host-side logic of the drop-in (module surface, state_dict compatibility, sharding
arithmetic, loud failure without CUDA)."""
import inspect

import pytest
import torch

import difformer
from difformer_b200 import ops
from difformer_b200.sharded import shard_rows
from tests.conftest import load_golden

MODEL = load_golden("model")
V2 = load_golden("v2")


def test_module_exports_reference_names():
    for name in ("DIFFormer", "DIFFormerConv", "full_attention_conv", "gcn_conv", "DIFFormer_v2", "TransConv"):
        assert hasattr(difformer, name)


def test_ctor_signature_matches_reference():
    # node classification/difformer.py:154-155
    sig = inspect.signature(difformer.DIFFormer.__init__)
    want = [("in_channels", inspect._empty), ("hidden_channels", inspect._empty), ("out_channels", inspect._empty),
            ("num_layers", 2), ("num_heads", 1), ("kernel", "simple"), ("alpha", 0.5), ("dropout", 0.5), ("use_bn", True),
            ("use_residual", True), ("use_weight", True), ("use_graph", True), ("graph_weight", -1), ("use_source", False)]
    got = [(n, p.default) for n, p in sig.parameters.items() if n != "self"]
    assert got == want
    sig2 = inspect.signature(difformer.DIFFormer_v2.__init__)     # difformer-v2.py:166-167
    got2 = [(n, p.default) for n, p in sig2.parameters.items() if n != "self"]
    assert got2 == [("in_channels", inspect._empty), ("hidden_channels", inspect._empty), ("out_channels", inspect._empty),
                    ("num_layers", 2), ("kernel", "simple"), ("alpha", 0.5), ("dropout", 0.5), ("use_bn", True),
                    ("use_residual", True), ("use_weight", True), ("use_graph", True), ("graph_weight", -1)]
    assert list(inspect.signature(difformer.DIFFormer.forward).parameters)[:4] == ["self", "x", "edge_index", "edge_weight"]
    assert list(inspect.signature(difformer.full_attention_conv).parameters)[:5] == ["qs", "ks", "vs", "kernel", "output_attn"]
    assert list(inspect.signature(difformer.gcn_conv).parameters)[:3] == ["x", "edge_index", "edge_weight"]


@pytest.mark.parametrize("name", sorted(MODEL))
def test_state_dict_round_trips_with_reference_checkpoints(name):
    c = MODEL[name]
    kw = {k[4:]: v for k, v in c.items() if k.startswith("cfg_")}
    for b in ("use_bn", "use_residual", "use_weight", "use_graph", "use_source"):
        if b in kw:
            kw[b] = bool(kw[b])
    m = difformer.DIFFormer(int(c["cin"]), int(c["hidden"]), int(c["cout"]), **kw)
    ref_sd = {k[3:]: v for k, v in c.items() if k.startswith("sd_")}
    assert sorted(m.state_dict().keys()) == sorted(ref_sd.keys())
    for k, v in m.state_dict().items():
        assert tuple(v.shape) == tuple(ref_sd[k].shape)
    m.load_state_dict(ref_sd, strict=True)      # test_large_dataset.py:86-88 does exactly this
    assert not list(m.buffers())                # no extra persistent state
    m.reset_parameters()


def test_v2_state_dict():
    c = V2["v2_model_simple"]
    m = difformer.DIFFormer_v2(16, 64, 3, num_layers=2)
    ref_sd = {k[3:]: v for k, v in c.items() if k.startswith("sd_")}
    assert sorted(m.state_dict().keys()) == sorted(ref_sd.keys())
    m.load_state_dict(ref_sd, strict=True)


def test_cpu_tensors_raise_instead_of_falling_back():
    q = torch.randn(8, 1, 64)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        difformer.full_attention_conv(q, q, q, "simple")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        difformer.full_attention_conv(q, q, q, "sigmoid")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        difformer.gcn_conv(q, torch.zeros(2, 4, dtype=torch.long), None)
    m = difformer.DIFFormer(8, 64, 3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(5, 8), torch.zeros(2, 4, dtype=torch.long))


def test_argument_validation():
    q = torch.randn(8, 2, 16)
    with pytest.raises(ValueError):
        ops._shapes(q, torch.randn(8, 3, 16), q)
    with pytest.raises(ValueError):
        ops._shapes(q, q, torch.randn(8, 3, 16))          # Hv must be H or 1
    assert ops._shapes(q, q, torch.randn(8, 1, 16)) == (8, 8, 2, 1, 16, 16)
    with pytest.raises(ValueError, match="unknown kernel"):
        difformer.full_attention_conv(q, q, q, "gaussian")
    with pytest.raises(TypeError):
        ops._f32c(q.double())


def test_shard_rows_partitions_exactly():
    for n in (0, 1, 7, 132534, 1632803):
        for world in (1, 2, 3, 4, 8):
            spans = [shard_rows(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            for (a, b), (c, d) in zip(spans, spans[1:]):
                assert b == c and a <= b
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_rows(10, 4, 4)


def test_seg_ptr_is_an_exclusive_scan():
    ptr = ops._seg_ptr(torch.tensor([5, 0, 17, 1]), 23, torch.device("cpu"))
    assert ptr.dtype == torch.int32 and ptr.tolist() == [0, 5, 5, 22, 23]


def test_epilogue_struct_layout():
    a = torch.zeros(4, 8)
    ep = ops.make_epilogue(0.125, [(a, 0.5), (a, 2.0)])
    assert ep.mode == 1 and ep.n_add == 2 and ep.add[0] == a.data_ptr() and abs(ep.add_scale[1] - 2.0) < 1e-7


def test_reference_parse_method_builds_this_model():
    """SURVEY 8b: the harness builds the model through `parse.parse_method` after `from difformer import *` (node
    classification/parse.py:2-10).  Replay the DIFFormer(...) calls the reference's own, unmodified parse.py makes on two command
    lines (recorded by oracle/make_golden.py, group parse_method) against this repo's `difformer` module: the object built must be
    this drop-in, with exactly the reference model's parameter names and shapes."""
    import json
    import os
    from tests.conftest import GOLDEN
    with open(os.path.join(GOLDEN, "parse_method.json")) as f:
        calls = json.load(f)
    assert len(calls) == 2
    for argv, call in calls.items():
        model = difformer.DIFFormer(*call["args"], **call["kwargs"]).to(torch.device("cpu"))
        assert type(model) is difformer.DIFFormer, argv
        got = {k: list(v.shape) for k, v in model.state_dict().items()}
        assert got == call["state_dict_shapes"], argv
        gen = torch.Generator().manual_seed(0)
        ref_sd = {k: torch.randn(shape, generator=gen) for k, shape in call["state_dict_shapes"].items()}
        model.load_state_dict(ref_sd)                      # checkpoints round-trip (test_large_dataset.py:86-88)
        assert all(torch.equal(model.state_dict()[k], t) for k, t in ref_sd.items())
        model.reset_parameters()                           # main.py:110


@pytest.mark.parametrize("h,use_weight", [(1, True), (2, False), (4, True)])
def test_projection_folding_algebra(h, use_weight):
    """SURVEY 8f-1 on the CPU: the operands `oracle.projected_operands` (the fp64 restatement of csrc/project.cu) derives from the Gram
    matrix X^T X, the column sums and the layer's weights reproduce full_attention_conv(Wq x, Wk x, Wv x, 'simple') exactly (fp64) --
    the algebra the GPU path rests on; the GPU tests check the kernel against this restatement."""
    from oracle import difformer_oracle as O
    torch.manual_seed(h)
    n = 700
    conv = difformer.DIFFormerConv(64, 64, num_heads=h, kernel="simple", use_weight=use_weight).double()
    with torch.no_grad():
        for p_ in conv.parameters():
            p_.mul_(3.0)
        x = torch.randn(n, 64, dtype=torch.float64) + 0.3
        G, s = x.t() @ x, x.sum(0)
        vpart, nvec, wbar, bbar = O.projected_operands(G, s, float(n), conv.Wq.weight, conv.Wq.bias, conv.Wk.weight, conv.Wk.bias,
                                                       conv.Wv.weight if use_weight else None, conv.Wv.bias if use_weight else None, h)
        A = vpart[:h * 4096].double().view(h, 64, 64)
        w = vpart[h * 4096:h * 4096 + h * 64].double().view(h, 64)
        u = vpart[h * 4096 + h * 64:h * 4096 + 2 * h * 64].double().view(h, 64)
        c = 1.0 / torch.sqrt(vpart[-2].double() * vpart[-1].double())
        num = c * torch.einsum("nc,hcd->nhd", x, A) + u.unsqueeze(0)
        den = c * torch.einsum("nc,hc->nh", x, w) + nvec.double().unsqueeze(0)
        got = num / den.unsqueeze(-1)
        q, k = conv.Wq(x).reshape(n, h, 64), conv.Wk(x).reshape(n, h, 64)
        v = conv.Wv(x).reshape(n, h, 64) if use_weight else x.reshape(n, 1, 64)
        want = O.simple_attention(q, k, v)
        assert O.rel_err(got, want) < 1e-10
        dev_part = want - want.mean(0, keepdim=True)            # mean-collapse guard: the part of the output that is not mean(V)
        assert O.rel_err(got - want.mean(0, keepdim=True), dev_part) < 1e-6
        vmean = v.mean(1) if use_weight else x
        assert O.rel_err(x @ wbar.double().t() + bbar.double(), vmean) < 1e-6


def test_segmented_tensor_core_dispatch_rules():
    """Host-side choice between the tensor-core tiles and the warp-per-graph kernels for the batched-graph 'simple' op (no GPU needed:
    the plan itself is only built when the rules say yes)."""
    class Lay:                       # what ops._seg_layout caches, minus the device plan
        def __init__(self, max_nodes, total):
            self.max_nodes, self.total, self.built = max_nodes, total, 0

        def plan(self):
            self.built += 1
            return "plan"
    try:
        ops.set_segmented_impl("auto")
        assert ops._segmented_tc_plan(Lay(40, 200000), 1, 1, 64, 64) == "plan"
        assert ops._segmented_tc_plan(Lay(40, 100), 1, 1, 64, 64) is None            # a handful of tiles: not worth it
        assert ops._segmented_tc_plan(Lay(90, 200000), 1, 1, 64, 64) is None          # tile fill below one half
        assert ops._segmented_tc_plan(Lay(40, 200000), 2, 2, 64, 64) is None          # one head only
        assert ops._segmented_tc_plan(Lay(40, 200000), 1, 1, 32, 32) is None          # hidden 64 only
        ops.set_segmented_impl("tcgen05")
        assert ops._segmented_tc_plan(Lay(128, 50), 1, 1, 64, 64) == "plan"           # pinned: whenever the shape allows
        assert ops._segmented_tc_plan(Lay(129, 5000), 1, 1, 64, 64) is None
        assert ops._segmented_tc_plan(Lay(0, 0), 1, 1, 64, 64) is None
        ops.set_segmented_impl("generic")
        lay = Lay(40, 200000)
        assert ops._segmented_tc_plan(lay, 1, 1, 64, 64) is None and lay.built == 0
        with pytest.raises(ValueError):
            ops.set_segmented_impl("fast")
    finally:
        ops.set_segmented_impl("auto")


def test_segmented_tile_plan_invariants():
    """The packing rule of the tensor-core batched-graph kernels (restated in oracle.segmented_tile_plan): for ANY batch layout with graphs
    of up to max_nodes <= 128 rows, tiles are whole graphs, at most 128 rows, in order, and cover every row exactly once."""
    from hypothesis import given, settings, strategies as st
    from oracle import difformer_oracle as O

    @settings(max_examples=150, deadline=None)
    @given(st.integers(1, 128).flatmap(lambda mx: st.tuples(st.just(mx), st.lists(st.integers(0, mx), min_size=1, max_size=120))))
    def check(arg):
        mx, sizes = arg
        n_nodes = torch.tensor(sizes)
        if int(n_nodes.sum()) == 0:
            return
        mx = max(int(n_nodes.max()), 1)
        tiles, rr = O.segmented_tile_plan(n_nodes, mx)
        N = int(n_nodes.sum())
        ptr = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(n_nodes.to(torch.int64), 0)])
        assert int(tiles[0]) == 0 and int(tiles[-1]) == N and int(tiles.min()) >= 0
        d = tiles[1:] - tiles[:-1]
        assert int(d.min()) >= 0 and int(d.max()) <= 128                      # ordered, at most 128 rows
        assert bool(torch.isin(tiles, ptr).all())                             # boundaries are graph boundaries
        nz = n_nodes > 0
        assert torch.equal(rr[:, 0], ptr[:-1][nz].repeat_interleave(n_nodes[nz]))
        assert torch.equal(rr[:, 1], ptr[1:][nz].repeat_interleave(n_nodes[nz]))
        if mx <= 64:                                                          # the regime the dispatcher picks: no empty tiles, fill >= 1/2 on average
            assert int(d[:-1].min()) > 0 if d.numel() > 1 else True
    check()

