"""CPU: pins oracle/difformer_oracle.py against the committed reference outputs (tests/golden,
made by oracle/make_golden.py from the unmodified reference).  Tolerances: 1e-5 rel in fp32 (pure reassociation noise),
2e-6 when the oracle runs in fp64 on the fp32 inputs."""
import filecmp
import json

import pytest
import torch

from oracle import difformer_oracle as O
from oracle import make_golden as G
from tests.conftest import load_golden

ATT = load_golden("attention")
GCN = load_golden("gcn")
MODEL = load_golden("model")
V2 = load_golden("v2")
RANDOM = load_golden("random_shapes")
PORT = load_golden("timing_port")


def _same_inputs(case, **tensors):
    """The inputs regenerated from their seeds are the ones the reference ran on (fp64 sums recorded with its outputs)."""
    for name, t in tensors.items():
        want = case["sum_" + name]
        assert abs(float(t.double().sum()) - want) <= 1e-9 * max(1.0, abs(want)), f"input {name} differs from the recorded one"


def _attn(name, c, dtype):
    q, k, v = (c[n].to(dtype) for n in "qkv")
    return (O.simple_attention if name.startswith("simple") else O.sigmoid_attention)(q, k, v)


@pytest.mark.parametrize("name", sorted(ATT))
def test_attention_forward_matches_reference_output(name):
    c = ATT[name]
    # nearly-centred V (the adversarial generator) amplifies fp32 summation noise in u = sum(V)
    tol = 2e-4 if abs(float(c["v"].mean())) < 0.05 else 1e-5
    assert O.rel_err(_attn(name, c, torch.float32), c["out"]) < tol
    assert O.rel_err(_attn(name, c, torch.float64), c["out"]) < tol


@pytest.mark.parametrize("name", sorted(ATT))
def test_attention_analytic_backward_matches_reference_autograd(name):
    c = ATT[name]
    bwd = O.simple_attention_backward if name.startswith("simple") else O.sigmoid_attention_backward
    dq, dk, dv = bwd(*(c[n].double() for n in "qkvg"))
    for got, want in ((dq, c["dq"]), (dk, c["dk"]), (dv, c["dv"])):
        assert O.rel_err(got, want) < 5e-5


@pytest.mark.parametrize("name", [n for n in sorted(ATT) if "attn" in ATT[n]])
def test_simple_dense_attention_branch(name):
    c = ATT[name]
    assert O.rel_err(O.simple_attention_dense_attn(c["q"], c["k"]), c["attn"]) < 1e-5


def test_simple_mean_collapse_is_real_and_intermediates_are_checked():
    """SURVEY.md 8a warning: `out` alone is dominated by mean(V); the term q^S^ must be pinned."""
    c = ATT["simple_n161_h4_d64"]
    out = O.simple_attention(c["q"], c["k"], c["v"])
    assert O.rel_err(c["v"].mean(0, keepdim=True).expand_as(out), out) < 1e-2     # collapse
    p = O.simple_partials(c["q"].double(), c["k"].double(), c["v"].double())
    _, parts = O.simple_apply(c["q"].double(), p, return_parts=True)
    # reconstruct the attention term from the reference output itself: out*den - u
    rec = c["out"].double() * parts["den"].unsqueeze(-1) - p["u"].unsqueeze(0)
    assert O.rel_err(rec, parts["qS"]) < 5e-2   # fp32 output only resolves the term to ~1e-2


@pytest.mark.parametrize("name", sorted(GCN))
def test_gcn_conv(name):
    c = GCN[name]
    out = O.gcn_conv(c["x"], c["edge_index"], c.get("edge_weight"))
    assert O.rel_err(out, c["out"]) < 1e-5
    if "dx" in c:
        assert O.rel_err(O.gcn_conv_backward_x(c["g"], c["edge_index"], c.get("edge_weight")), c["dx"]) < 1e-5


def _model_kwargs(c):
    kw = {k[4:]: v for k, v in c.items() if k.startswith("cfg_")}
    for b in ("use_bn", "use_residual", "use_weight", "use_graph", "use_source"):
        if b in kw:
            kw[b] = bool(kw[b])
    return kw


@pytest.mark.parametrize("name", sorted(MODEL))
def test_model_forward(name):
    c = MODEL[name]
    sd = {k[3:]: v for k, v in c.items() if k.startswith("sd_")}
    out = O.difformer_forward(sd, c["x"], c["edge_index"], c.get("edge_weight"),
                              hidden_channels=int(c["hidden"]), **_model_kwargs(c))
    assert O.rel_err(out, c["out"]) < 2e-5


def test_v2_segmented_simple():
    for name in ("v2_simple_segments", "v2_simple_segments_h2"):
        c = V2[name]
        assert O.rel_err(O.segmented_simple_attention(c["q"], c["k"], c["v"], c["n_nodes"]), c["out"]) < 1e-5
    c = V2["v2_simple_segments"]
    dq, dk, dv = O.segmented_simple_attention_backward(*(c[n].double() for n in "qkv"), c["n_nodes"], c["g"].double())
    for got, want in ((dq, c["dq"]), (dk, c["dk"]), (dv, c["dv"])):
        assert O.rel_err(got, want) < 5e-5


def test_v2_model_forward():
    c = V2["v2_model_simple"]
    sd = {k[3:]: v for k, v in c.items() if k.startswith("sd_")}
    out = O.difformer_v2_forward(sd, c["x"], c["edge_index"], c["n_nodes"], hidden_channels=64)
    assert O.rel_err(out, c["out"]) < 2e-5


def test_oracle_against_live_reference_random_shapes():
    """The oracle against the reference's outputs on seeded random shapes (edge cases N = 1 and Hv = 1 < H included), recorded by
    oracle/make_golden.py (group random_shapes) on a sample of the output rows."""
    for n, h, d, hv, q, k, v, ei, w in G.random_shape_inputs():
        c = RANDOM[f"shape_n{n}_h{h}_d{d}_hv{hv}"]
        _same_inputs(c, q=q, k=k, v=v, edge_index=ei, edge_weight=w)
        rows = c["rows"]
        # nearly-centred V amplifies fp32 summation noise; the fp64 arbiter below is tight
        assert O.rel_err(O.simple_attention(q, k, v)[rows], c["simple"]) < 2e-4
        assert O.rel_err(O.sigmoid_attention(q * .2, k * .2, v)[rows], c["sigmoid"]) < 1e-5
        assert O.rel_err(O.gcn_conv(v, ei, w)[rows], c["gcn"]) < 1e-5
        # fp64 arbiter
        assert O.rel_err(O.simple_attention(q.double(), k.double(), v.double())[rows], c["simple64"]) < 1e-12
    c = RANDOM["segmented"]
    q, k, v, nn_ = G.segmented_inputs()
    _same_inputs(c, q=q, k=k, v=v)
    assert torch.equal(nn_, c["n_nodes"])
    assert O.rel_err(O.segmented_simple_attention(q, k, v, nn_), c["out"]) < 1e-5


def test_timing_port_is_bit_equal_to_the_reference_function():
    """`bench.py`'s CPU baseline times the real `full_attention_conv` when oracle/_ref exists and this port of it otherwise:
    the port must compute exactly the reference's values.  It runs the reference's op chain -- the same aten ops on the same
    shapes and dtypes, in the same order, hence the same values bit for bit on any one machine -- and its output matches the
    reference's recorded output to fp32 reassociation noise (the recording machine's thread count and vector ISA set the last bits)."""
    for n, h, d in G.TIMING_PORT_SHAPES:
        c = PORT[f"n{n}_h{h}_d{d}"]
        q, k, v = O.synthetic_qkv(n, h, d, seed=n)
        _same_inputs(c, q=q, k=k, v=v)
        assert G.op_chain(O.simple_attention_reference_chain, q, k, v) == json.loads(c["op_chain"])
        assert O.rel_err(O.simple_attention_reference_chain(q, k, v)[c["rows"]], c["out"]) < 1e-5


def test_vendored_reference_is_a_byte_copy(tmp_path, monkeypatch):
    """oracle/build_ref.py (which fills the git-ignored oracle/_ref) must copy the reference files unmodified, and keep an earlier
    copy when the reference tree is absent.  Checked on a stand-in tree of the same layout."""
    from oracle import build_ref as B
    src, dst = tmp_path / "src", tmp_path / "dst"
    for i, rel in enumerate(B.FILES):
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_bytes(bytes(range(256)) * (i + 3) + b"\r\n\x00 trailing bytes without a newline")
    monkeypatch.setattr(B, "SRC", str(src))
    monkeypatch.setattr(B, "DST", str(dst))
    assert B.build_ref(verbose=False)
    for rel in B.FILES:
        assert filecmp.cmp(str(src / rel), str(dst / rel), shallow=False)
    monkeypatch.setattr(B, "SRC", str(tmp_path / "absent"))
    assert not B.build_ref(verbose=False)
    for rel in B.FILES:
        assert filecmp.cmp(str(src / rel), str(dst / rel), shallow=False)


def test_v2_sigmoid_oracle_matches_reference_golden():
    """a-7: the slot-by-slot restatement of the batched 'sigmoid' (difformer-v2.py:113-135) against the reference's outputs."""
    v2 = load_golden("v2")
    for name in ("v2_sigmoid_segments", "v2_sigmoid_segments_h2"):
        c = v2[name]
        got = O.segmented_sigmoid_attention(c["q"], c["k"], c["v"], c["n_nodes"])
        assert O.rel_err(got, c["out"]) < 1e-5, name
        q, k, v = (c[n].double().requires_grad_(True) for n in ("q", "k", "v"))     # autograd of the restatement = the reference's grads
        O.segmented_sigmoid_attention(q, k, v, c["n_nodes"]).backward(c["g"].double())
        for got_g, want in ((q.grad, c["dq"]), (k.grad, c["dk"]), (v.grad, c["dv"])):
            assert O.rel_err(got_g, want) < 1e-4, name
