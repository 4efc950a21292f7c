"""TEST INFRASTRUCTURE -- generates tests/golden/* by running the UNMODIFIED reference
(`node classification/difformer.py`, `node classification/parse.py`, `physical particle/difformer-v2.py`) under
`oracle/ref_shim.py`.  Needs a checkout of the reference project:

    python oracle/make_golden.py                      # every group
    python oracle/make_golden.py random_shapes ...    # only the named groups (the others stay byte-identical)

The reference has no golden vectors of its own (SURVEY.md section 8c), so these fixtures -- outputs of
the reference code itself on seeded inputs -- are what pins both the oracle restatement and the
CUDA path.  torch 2.11.0 CPU, fp32, seeds listed per case.
"""
import argparse
import importlib.util
import json
import os
import sys
import types

import numpy as np
import torch
from torch.utils._python_dispatch import TorchDispatchMode

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.difformer_oracle import synthetic_graph, synthetic_qkv  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# shapes (N, H, D, Hv) of the randomised oracle-vs-reference check, edge cases included (N = 1, Hv = 1 < H)
RANDOM_SHAPES = [(50, 1, 8, 1), (200, 4, 64, 4), (77, 3, 16, 1), (1, 2, 4, 2), (513, 2, 32, 2)]
# (N, H, D) of the check that bench.py's CPU baseline port runs the reference's own op chain
TIMING_PORT_SHAPES = [(300, 4, 64), (129, 1, 32)]
# command lines the reference harness (node classification/parse.py) is run with to build a DIFFormer
PARSE_ARGVS = [["--use_bn", "--use_residual", "--use_graph", "--hidden_channels", "64"],
               ["--use_bn", "--use_residual", "--use_graph", "--use_weight", "--use_source", "--num_heads", "4", "--kernel", "sigmoid",
                "--hidden_channels", "32", "--num_layers", "3", "--graph_weight", "0.5"]]
PARSE_SIZES = (100, 7, 33)          # parse_method(args, n, c, d, device): nodes, classes, input features


def sample_rows(n, k=16, seed=0):
    """Rows of an output that a fixture keeps: all of them up to 64, else k rows drawn once with a fixed seed (keeps the files small;
    the inputs are regenerated from their seeds, so every row still takes part in the computation)."""
    if n <= 64:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:k].sort().values


def random_shape_inputs():
    """Yields (n, h, d, hv, q, k, v, edge_index, edge_weight) for RANDOM_SHAPES: seeded, identical on every run."""
    gen = torch.Generator().manual_seed(0)
    for n, h, d, hv in RANDOM_SHAPES:
        q, k, v = synthetic_qkv(n, h, d, seed=n, hv=hv, adversarial=True)
        ei = torch.randint(0, n, (2, 5 * n), generator=gen)
        w = torch.rand(5 * n, generator=gen)
        yield n, h, d, hv, q, k, v, ei, w


def segmented_inputs():
    """The batched-graph case of the randomised check: four graphs of 3, 10, 1 and 25 nodes, H = 1, D = 16."""
    q, k, v = synthetic_qkv(39, 1, 16, seed=4)
    return q, k, v, torch.tensor([3, 10, 1, 25])


def input_fingerprint(**tensors):
    """fp64 sums of the inputs: a test that regenerates them from their seeds checks it has the ones the reference saw."""
    return {"sum_" + name: np.float64(t.double().sum()) for name, t in tensors.items()}


def random_shape_cases(ref, ref2):
    cases = {}
    for n, h, d, hv, q, k, v, ei, w in random_shape_inputs():
        rows = sample_rows(n)
        qd, kd, vd = q.double(), k.double(), v.double()
        torch.set_default_dtype(torch.float64)      # the reference builds its `ones` in the default dtype
        try:
            simple64 = ref.full_attention_conv(qd, kd, vd, "simple")
        finally:
            torch.set_default_dtype(torch.float32)
        cases[f"shape_n{n}_h{h}_d{d}_hv{hv}"] = _np(dict(
            rows=rows, simple=ref.full_attention_conv(q, k, v, "simple")[rows],
            sigmoid=ref.full_attention_conv(q * .2, k * .2, v, "sigmoid")[rows],
            gcn=ref.gcn_conv(v, ei, w)[rows], simple64=simple64[rows],
            **input_fingerprint(q=q, k=k, v=v, edge_index=ei, edge_weight=w)))
    q, k, v, nn_ = segmented_inputs()
    cases["segmented"] = _np(dict(out=ref2.TransConv(16, 16).full_attention(q, k, v, "simple", nn_), n_nodes=nn_,
                                  **input_fingerprint(q=q, k=k, v=v)))
    return cases


class OpChain(TorchDispatchMode):
    """Records the aten ops a function runs, as (op, output shape, output dtype).  In-place and out-of-place forms of an op are
    recorded alike (`x += y` and `x = x + y` compute the same values), and the constant factories `ones` / `ones_like` are left out
    (the reference builds the same all-ones vector twice)."""
    FACTORIES = ("ones", "ones_like")

    def __init__(self):
        super().__init__()
        self.ops = []

    def __torch_dispatch__(self, func, types_, args=(), kwargs=None):
        out = func(*args, **(kwargs or {}))
        name = func.overloadpacket.__name__.rstrip("_")
        if name not in self.FACTORIES:
            outs = out if isinstance(out, (tuple, list)) else (out,)
            self.ops.append([name] + [[list(t.shape), str(t.dtype).replace("torch.", "")] if torch.is_tensor(t) else repr(t) for t in outs])
        return out


def op_chain(fn, *args):
    with OpChain() as rec:
        fn(*args)
    return rec.ops


def timing_port_cases(ref):
    """The reference's `full_attention_conv(.., 'simple')` on TIMING_PORT_SHAPES: its op chain (a JSON string) and a sample of its
    output rows."""
    cases = {}
    for n, h, d in TIMING_PORT_SHAPES:
        q, k, v = synthetic_qkv(n, h, d, seed=n)
        rows = sample_rows(n)
        cases[f"n{n}_h{h}_d{d}"] = _np(dict(op_chain=np.array(json.dumps(op_chain(ref.full_attention_conv, q, k, v, "simple"))), rows=rows,
                                            out=ref.full_attention_conv(q, k, v, "simple")[rows], **input_fingerprint(q=q, k=k, v=v)))
    return cases


def parse_method_cases(ref):
    """How the reference harness builds the model: run its own parse.py on PARSE_ARGVS with a stand-in `difformer` module that records
    the DIFFormer(...) call, and the parameter shapes of the reference DIFFormer that call builds."""
    from oracle.ref_shim import REFERENCE_ROOT
    calls = []

    class Recorder:
        def __init__(self, *args, **kwargs):
            calls.append((list(args), kwargs))

        def to(self, device):
            return self
    saved = {k: sys.modules.get(k) for k in ("gnns", "difformer")}
    sys.modules["gnns"] = types.ModuleType("gnns")          # baseline GNN zoo (PyG): out of scope, star-import of an empty module
    stub = types.ModuleType("difformer")
    stub.DIFFormer = Recorder
    sys.modules["difformer"] = stub
    try:
        spec = importlib.util.spec_from_file_location("_reference_parse", os.path.join(REFERENCE_ROOT, "node classification", "parse.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        cases = {}
        for argv in PARSE_ARGVS:
            parser = argparse.ArgumentParser()
            mod.parser_add_main_args(parser)
            mod.parse_method(parser.parse_args(argv), *PARSE_SIZES, torch.device("cpu"))
            args, kwargs = calls.pop()
            model = ref.DIFFormer(*args, **kwargs)
            cases[" ".join(argv)] = {"args": args, "kwargs": kwargs,
                                     "state_dict_shapes": {k: list(t.shape) for k, t in model.state_dict().items()}}
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return cases


def _np(d):
    return {k: (v.detach().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in d.items()}


def attention_cases(ref):
    cases = {}
    specs = [  # name, kernel, N, H, D, Hv, adversarial, seed
        ("simple_n161_h4_d64", "simple", 161, 4, 64, 4, False, 123),
        ("simple_n140_h4_d64_adv", "simple", 140, 4, 64, 4, True, 7),
        ("simple_n64_h1_d64", "simple", 64, 1, 64, 1, False, 11),
        ("simple_n129_h2_d32_hv1", "simple", 129, 2, 32, 1, True, 5),
        ("simple_n33_h3_d16", "simple", 33, 3, 16, 3, True, 9),
        ("sigmoid_n150_h1_d64", "sigmoid", 150, 1, 64, 1, False, 123),
        ("sigmoid_n101_h4_d64", "sigmoid", 101, 4, 64, 4, True, 3),
        ("sigmoid_n77_h2_d32_hv1", "sigmoid", 77, 2, 32, 1, False, 21),
    ]
    for name, kernel, n, h, d, hv, adv, seed in specs:
        q, k, v = synthetic_qkv(n, h, d, seed=seed, hv=hv, adversarial=adv)
        if kernel == "sigmoid":
            q, k = q * 0.3, k * 0.3
        q, k, v = (t.clone().requires_grad_(True) for t in (q, k, v))
        out = ref.full_attention_conv(q, k, v, kernel)
        g = torch.randn(out.shape, generator=torch.Generator().manual_seed(seed + 1000))
        out.backward(g)
        cases[name] = _np(dict(q=q, k=k, v=v, out=out, g=g, dq=q.grad, dk=k.grad, dv=v.grad))
        if kernel == "simple" and h == 1:  # :43 only broadcasts correctly for H == 1
            _, att = ref.full_attention_conv(q.detach(), k.detach(), v.detach(), kernel, output_attn=True)
            cases[name]["attn"] = att.numpy()
    return cases


def gcn_cases(ref):
    cases = {}
    # (a) undirected + self loops, no weights  (what main.py:72-79 feeds)
    n = 150
    ei = synthetic_graph(n, 400, seed=1)
    x = torch.randn(n, 4, 64, generator=torch.Generator().manual_seed(2))
    cases["gcn_undirected_selfloops"] = _np(dict(x=x, edge_index=ei, out=ref.gcn_conv(x, ei, None)))
    # (b) directed, duplicates, isolated nodes, sources with zero in-degree (-> inf -> 0), weights incl. 0/NaN/inf
    gen = torch.Generator().manual_seed(3)
    n = 97
    row = torch.randint(0, n, (500,), generator=gen)
    col = torch.randint(0, n // 2, (500,), generator=gen)      # upper half never a target: d=0 there
    row[:20], col[:20] = row[20:40], col[20:40]                # exact duplicates
    ei = torch.stack([row, col])
    w = torch.rand(500, generator=gen) * 2 - 0.5
    w[5], w[6], w[7] = 0.0, float("nan"), float("inf")
    x = torch.randn(n, 1, 32, generator=gen)
    cases["gcn_directed_weighted"] = _np(dict(x=x, edge_index=ei, edge_weight=w, out=ref.gcn_conv(x, ei, w)))
    cases["gcn_directed_unweighted"] = _np(dict(x=x, edge_index=ei, out=ref.gcn_conv(x, ei, None)))
    # (c) backward through gcn_conv wrt x
    xg = torch.randn(n, 2, 16, generator=gen).requires_grad_(True)
    out = ref.gcn_conv(xg, ei, w)
    g = torch.randn(out.shape, generator=gen)
    out.backward(g)
    cases["gcn_backward"] = _np(dict(x=xg, edge_index=ei, edge_weight=w, out=out, g=g, dx=xg.grad))
    return cases


def model_cases(ref):
    cases = {}
    specs = [  # name, ctor kwargs, N, C_in, C_out, n_pairs, edge weights?
        ("model_simple_cora_like", dict(num_layers=2, num_heads=1, kernel="simple", use_bn=True, use_residual=True,
                                        use_weight=False, use_graph=True), 120, 40, 7, 300, False),
        ("model_simple_h4_weight_source", dict(num_layers=2, num_heads=4, kernel="simple", use_bn=True, use_residual=True,
                                               use_weight=True, use_graph=True, graph_weight=0.3, use_source=True), 90, 24, 5, 200, True),
        ("model_simple_nograph_nobn", dict(num_layers=3, num_heads=2, kernel="simple", use_bn=False, use_residual=False,
                                           use_weight=True, use_graph=False, alpha=0.7), 75, 12, 3, 100, False),
        ("model_sigmoid_h2", dict(num_layers=2, num_heads=2, kernel="sigmoid", use_bn=True, use_residual=True,
                                  use_weight=True, use_graph=True), 83, 20, 4, 150, False),
    ]
    for name, kw, n, cin, cout, pairs, weighted in specs:
        torch.manual_seed(123)
        hid = 64
        m = ref.DIFFormer(cin, hid, cout, **kw)
        m.eval()
        gen = torch.Generator().manual_seed(77)
        x = torch.randn(n, cin, generator=gen)
        ei = synthetic_graph(n, pairs, seed=5)
        w = torch.rand(ei.shape[1], generator=gen) + 0.5 if weighted else None
        # train-mode-free backward: eval mode so dropout is the identity, grads are deterministic
        out = m(x, ei, w) if weighted else m(x, ei)
        loss = (out * torch.randn(out.shape, generator=gen)).sum()
        loss.backward()
        d = dict(x=x, edge_index=ei, out=out, hidden=hid, cin=cin, cout=cout)
        if weighted:
            d["edge_weight"] = w
        for k_, v_ in kw.items():
            d["cfg_" + k_] = v_
        for k_, v_ in m.state_dict().items():
            d["sd_" + k_] = v_
        for k_, p in m.named_parameters():
            if p.grad is not None:          # use_bn=False leaves the LayerNorms unused
                d["grad_" + k_] = p.grad
        cases[name] = _np(d)
    return cases


def v2_cases(ref2):
    cases = {}
    gen = torch.Generator().manual_seed(31)
    n_nodes = torch.tensor([5, 17, 1, 40, 23, 9])
    tot = int(n_nodes.sum())
    q, k, v = (torch.randn(tot, 1, 64, generator=gen) + 0.3 for _ in range(3))
    conv = ref2.TransConv(64, 64)
    q, k, v = (t.clone().requires_grad_(True) for t in (q, k, v))
    out = conv.full_attention(q, k, v, "simple", n_nodes)
    g = torch.randn(out.shape, generator=gen)
    out.backward(g)
    cases["v2_simple_segments"] = _np(dict(q=q, k=k, v=v, n_nodes=n_nodes, out=out, g=g, dq=q.grad, dk=k.grad, dv=v.grad))
    # multi-head variant (the class never uses it, the function supports it)
    q, k, v = (torch.randn(tot, 2, 32, generator=gen) for _ in range(3))
    cases["v2_simple_segments_h2"] = _np(dict(q=q, k=k, v=v, n_nodes=n_nodes,
                                              out=conv.full_attention(q, k, v, "simple", n_nodes)))
    # whole model, eval mode
    torch.manual_seed(123)
    m = ref2.DIFFormer_v2(16, 64, 3, num_layers=2, kernel="simple", use_graph=True)
    m.eval()
    x = torch.randn(tot, 16, generator=gen)
    # block-diagonal edges: ring inside each graph + self loops
    rows, cols, s = [], [], 0
    for n in n_nodes.tolist():
        idx = torch.arange(n) + s
        rows += [idx, idx.roll(1), idx]
        cols += [idx.roll(1), idx, idx]
        s += n
    ei = torch.stack([torch.cat(rows), torch.cat(cols)])
    out = m(x, ei, n_nodes)
    d = dict(x=x, edge_index=ei, n_nodes=n_nodes, out=out)
    for k_, v_ in m.state_dict().items():
        d["sd_" + k_] = v_
    cases["v2_model_simple"] = _np(d)
    # kernel='sigmoid' of the batched variant (difformer-v2.py:113-135): cross-graph attention between the nodes that share
    # a padded slot; appended last so that the random draws of the cases above stay what they were
    gen2 = torch.Generator().manual_seed(77)
    nn2 = torch.tensor([4, 9, 1, 12, 7])
    tot2 = int(nn2.sum())
    for name, h, d, scale in (("v2_sigmoid_segments", 1, 64, 0.3), ("v2_sigmoid_segments_h2", 2, 32, 0.5)):
        q, k, v = (torch.randn(tot2, h, d, generator=gen2) * s_ for s_ in (scale, scale, 1.0))
        q, k, v = (t.clone().requires_grad_(True) for t in (q, k, v))
        out = conv.full_attention(q, k, v, "sigmoid", nn2)
        g = torch.randn(out.shape, generator=gen2)
        out.backward(g)
        cases[name] = _np(dict(q=q, k=k, v=v, n_nodes=nn2, out=out, g=g, dq=q.grad, dk=k.grad, dv=v.grad))
    return cases


NPZ_GROUPS = {"attention": lambda ref, ref2: attention_cases(ref), "gcn": lambda ref, ref2: gcn_cases(ref),
              "model": lambda ref, ref2: model_cases(ref), "v2": lambda ref, ref2: v2_cases(ref2),
              "random_shapes": random_shape_cases, "timing_port": lambda ref, ref2: timing_port_cases(ref)}
JSON_GROUPS = {"parse_method": lambda ref, ref2: parse_method_cases(ref)}


def main(names):
    unknown = set(names) - set(NPZ_GROUPS) - set(JSON_GROUPS)
    if unknown:
        raise SystemExit(f"unknown group(s) {sorted(unknown)}; known: {list(NPZ_GROUPS) + list(JSON_GROUPS)}")
    from oracle.ref_shim import load_reference_v1, load_reference_v2      # here, not at import: the tests import this module
    os.makedirs(OUT, exist_ok=True)
    ref, ref2 = load_reference_v1(), load_reference_v2()
    for gname in names or list(NPZ_GROUPS) + list(JSON_GROUPS):
        cases = (NPZ_GROUPS.get(gname) or JSON_GROUPS[gname])(ref, ref2)
        if gname in NPZ_GROUPS:
            flat = {}
            for cname, arrs in cases.items():
                for k, v in arrs.items():
                    flat[f"{cname}/{k}"] = v
            path = os.path.join(OUT, f"{gname}.npz")
            np.savez_compressed(path, **flat)
        else:
            path = os.path.join(OUT, f"{gname}.json")
            with open(path, "w") as f:
                json.dump(cases, f, indent=1)
                f.write("\n")
        print(f"{path}: {len(cases)} cases, {os.path.getsize(path) / 1e3:.0f} kB")


if __name__ == "__main__":
    main(sys.argv[1:])
