"""CPU ORACLE -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

An independent CPU restatement (torch CPU tensors, dtype-generic so the same code is the fp64
arbiter) of the one DIFFormer hot path this repo accelerates.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` legs may import this
file; `difformer_b200/` never does (the product path has no CPU fallback and raises when the CUDA
library is missing).

Pinning: the reference ships no tests or golden vectors (SURVEY.md section 4/8c).  This restatement is
pinned against the reference *itself*: `oracle/make_golden.py` runs the unmodified reference
files (under `oracle/ref_shim.py`) in the build container and commits input/output vectors to
`tests/golden/`; `tests/test_oracle_golden.py` checks every function below against those
vectors.  All line citations are relative to the root of the reference project.

Algebra is written in matmul/reduction form on purpose (the reference uses einsum chains and
materialises broadcasts) so agreement is a meaningful check of the algorithm, not of a copy.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch

Tensor = torch.Tensor


# --------------------------------------------------------------------------------------------
# a-1  kernel='simple'     node classification/difformer.py:18-39
# --------------------------------------------------------------------------------------------
def simple_partials(qs: Tensor, ks: Tensor, vs: Tensor) -> Dict[str, Tensor]:
    """Un-normalised row reductions of pass 1 (what one row shard contributes to the all-reduce).

    S[h,m,d] = sum_l k[l,h,m] v[l,hv,d]    (difformer.py:25 before the 1/||K|| scale)
    z[h,m]   = sum_l k[l,h,m]              (difformer.py:32-33)
    u[hv,d]  = sum_l v[l,hv,d]             (difformer.py:27-28)
    sq, sk   = sum q^2, sum k^2            (difformer.py:20-21, squared Frobenius norms)
    V may carry one head (use_weight=False, difformer.py:120) -- it broadcasts over H.
    """
    H, Hv = ks.shape[1], vs.shape[1]
    vb = vs if Hv == H else vs.expand(-1, H, -1)
    S = torch.matmul(ks.permute(1, 2, 0), vb.permute(1, 0, 2))          # [H,M,L]x[H,L,D]
    return {"S": S, "z": ks.sum(0), "u": vs.sum(0), "sq": (qs * qs).sum(), "sk": (ks * ks).sum(),
            "n": torch.tensor(float(ks.shape[0]), dtype=qs.dtype)}


def simple_apply(qs: Tensor, p: Dict[str, Tensor], n_total: Optional[float] = None,
                 return_parts: bool = False):
    """Pass 2: out = (q^ S^ + u) / (q^ z^ + N), difformer.py:26,29,34,37-39.

    q^ = q/||Q||_F, S^ = S/||K||_F, z^ = z/||K||_F.  The normaliser N is the number of *source*
    rows (difformer.py:22 uses qs.shape[0], and :29 requires N == L).
    """
    n = float(p["n"]) if n_total is None else float(n_total)
    c = 1.0 / (torch.sqrt(p["sq"]) * torch.sqrt(p["sk"]))
    qS = torch.matmul(qs.permute(1, 0, 2), p["S"]).permute(1, 0, 2) * c   # [N,H,D]
    qz = (qs * p["z"].unsqueeze(0)).sum(-1) * c                           # [N,H]
    num = qS + p["u"].unsqueeze(0)
    den = qz + n
    out = num / den.unsqueeze(-1)
    if return_parts:
        return out, {"qS": qS, "qz": qz, "num": num, "den": den}
    return out


def simple_attention(qs: Tensor, ks: Tensor, vs: Tensor) -> Tensor:
    """full_attention_conv(qs, ks, vs, 'simple')  -- difformer.py:10-39,58-61."""
    return simple_apply(qs, simple_partials(qs, ks, vs))


def simple_attention_reference_chain(qs: Tensor, ks: Tensor, vs: Tensor) -> Tensor:
    """Op-for-op transcription of the reference's einsum chain (difformer.py:18-39), including its
    materialised broadcasts (`repeat`, `ones`), for TIMING the "reference PyTorch path" on CPU or on
    the same GPU (BASELINE.md section 4 item 2).  Same maths as `simple_attention`; kept separate because
    the launch count / memory traffic of this exact chain is what the speed-up is quoted against."""
    qs = qs / torch.norm(qs, p=2)                                                    # :20
    ks = ks / torch.norm(ks, p=2)                                                    # :21
    n = qs.shape[0]
    kvs = torch.einsum("lhm,lhd->hmd", ks, vs)                                       # :25
    num = torch.einsum("nhm,hmd->nhd", qs, kvs)                                      # :26
    ones = torch.ones([vs.shape[0]], device=vs.device, dtype=vs.dtype)               # :27
    vs_sum = torch.einsum("l,lhd->hd", ones, vs)                                     # :28
    num = num + vs_sum.unsqueeze(0).repeat(vs.shape[0], 1, 1)                        # :29
    ks_sum = torch.einsum("lhm,l->hm", ks, ones)                                     # :33
    den = torch.einsum("nhm,hm->nh", qs, ks_sum).unsqueeze(-1)                       # :34,37
    den = den + torch.ones_like(den) * n                                             # :38
    return num / den                                                                 # :39


def simple_attention_dense_attn(qs: Tensor, ks: Tensor) -> Tensor:
    """output_attn branch, difformer.py:42-43: q^k^T/den WITHOUT the '+1' (rows do not sum to 1)."""
    a, b = torch.linalg.vector_norm(qs), torch.linalg.vector_norm(ks)
    qh, kh = qs / a, ks / b
    den = (qh * kh.sum(0).unsqueeze(0)).sum(-1) + qs.shape[0]             # [N,H]
    att = torch.matmul(qh.permute(1, 0, 2), kh.permute(1, 2, 0)).permute(1, 2, 0)  # [N,L,H]
    return att / den.unsqueeze(1)


def simple_attention_backward(qs: Tensor, ks: Tensor, vs: Tensor, g: Tensor
                              ) -> Tuple[Tensor, Tensor, Tensor]:
    """Analytic backward of a-1 (SURVEY.md section 8a-1b; the reference relies on autograd)."""
    H, Hv = ks.shape[1], vs.shape[1]
    a, b = torch.linalg.vector_norm(qs), torch.linalg.vector_norm(ks)
    qh, kh = qs / a, ks / b
    vb = vs if Hv == H else vs.expand(-1, H, -1)
    S = torch.matmul(kh.permute(1, 2, 0), vb.permute(1, 0, 2))            # [H,M,D]
    z = kh.sum(0)
    den = (qh * z.unsqueeze(0)).sum(-1) + qs.shape[0]                     # [N,H]
    out = (torch.matmul(qh.permute(1, 0, 2), S).permute(1, 0, 2) + vb.sum(0).unsqueeze(0)) / den.unsqueeze(-1)
    dnum = g / den.unsqueeze(-1)                                          # [N,H,D]
    dden = -(g * out).sum(-1) / den                                       # [N,H]
    dqh = torch.matmul(dnum.permute(1, 0, 2), S.transpose(1, 2)).permute(1, 0, 2) + dden.unsqueeze(-1) * z.unsqueeze(0)
    dS = torch.matmul(qh.permute(1, 2, 0), dnum.permute(1, 0, 2))         # [H,M,D]
    dz = (qh * dden.unsqueeze(-1)).sum(0)                                 # [H,M]
    du = dnum.sum(0)                                                      # [H,D]
    dkh = torch.matmul(vb.permute(1, 0, 2), dS.transpose(1, 2)).permute(1, 0, 2) + dz.unsqueeze(0)
    dvb = torch.matmul(kh.permute(1, 0, 2), dS).permute(1, 0, 2) + du.unsqueeze(0)
    dv = dvb if Hv == H else dvb.sum(1, keepdim=True)
    dq = (dqh - qh * (qh * dqh).sum()) / a
    dk = (dkh - kh * (kh * dkh).sum()) / b
    return dq, dk, dv


# --------------------------------------------------------------------------------------------
# a-2  kernel='sigmoid'    node classification/difformer.py:45-56
# --------------------------------------------------------------------------------------------
def sigmoid_attention(qs: Tensor, ks: Tensor, vs: Tensor, return_rowsum: bool = False):
    """P = sigmoid(q.k) with no 1/sqrt(d) and no normalisation (:47); r = row sums (:50-51);
    out = (P/r) V (:55-56).  Evaluated head by head, never materialising [N,L,H]."""
    N, H, _ = qs.shape
    Hv = vs.shape[1]
    out = qs.new_empty(N, H, vs.shape[2])
    rs = qs.new_empty(N, H)
    for h in range(H):
        P = torch.sigmoid(qs[:, h] @ ks[:, h].T)
        r = P.sum(1)
        out[:, h] = (P @ vs[:, h if Hv == H else 0]) / r.unsqueeze(1)
        rs[:, h] = r
    return (out, rs) if return_rowsum else out


def sigmoid_attention_backward(qs: Tensor, ks: Tensor, vs: Tensor, g: Tensor):
    """Analytic backward of a-2 (SURVEY.md section 8a-2b)."""
    N, H, _ = qs.shape
    Hv = vs.shape[1]
    dq, dk = torch.zeros_like(qs), torch.zeros_like(ks)
    dv = torch.zeros_like(vs)
    for h in range(H):
        hv = h if Hv == H else 0
        P = torch.sigmoid(qs[:, h] @ ks[:, h].T)
        r = P.sum(1, keepdim=True)
        A = P / r
        out = A @ vs[:, hv]
        dv[:, hv] += A.T @ g[:, h]
        dA = g[:, h] @ vs[:, hv].T
        dP = (dA - (g[:, h] * out).sum(1, keepdim=True)) / r
        dSc = dP * P * (1 - P)
        dq[:, h] = dSc @ ks[:, h]
        dk[:, h] = dSc.T @ qs[:, h]
    return dq, dk, dv


# --------------------------------------------------------------------------------------------
# a-3  gcn_conv            node classification/difformer.py:63-79
# --------------------------------------------------------------------------------------------
def gcn_edge_values(edge_index: Tensor, edge_weight: Optional[Tensor], n: int,
                    dtype=torch.float32) -> Tensor:
    """val_e = w_e * d[col_e]^-1/2 * d[row_e]^-1/2 with d = in-degree histogram of `col` for BOTH
    factors (:66-68); w=1 when None (:70-73); non-finite -> 0 (:74).  torch_geometric.utils.degree
    1.7.2 = scatter-add of ones.  The degree arithmetic is float32 in the reference (:66 .float())."""
    row, col = edge_index[0].long(), edge_index[1].long()
    d = torch.bincount(col, minlength=n).to(torch.float32)
    d_in, d_out = (1.0 / d[col]).sqrt(), (1.0 / d[row]).sqrt()
    # same association as the reference: (w * d_in) * d_out, w = 1 when absent (:70-73)
    val = (edge_weight.to(torch.float32) * d_in if edge_weight is not None else d_in) * d_out
    val = torch.where(torch.isfinite(val), val, torch.zeros_like(val))
    return val.to(dtype)


def gcn_conv(x: Tensor, edge_index: Tensor, edge_weight: Optional[Tensor]) -> Tensor:
    """out[c,h,:] = sum_{e: col_e = c} val_e * x[row_e,h,:]  (:75-78; torch_sparse 0.6.10
    SparseTensor(row=col, col=row) + matmul(reduce='sum'): duplicates are summed)."""
    n = x.shape[0]
    val = gcn_edge_values(edge_index, edge_weight, n, x.dtype)
    out = torch.zeros_like(x)
    out.index_add_(0, edge_index[1].long(), val.view(-1, 1, 1) * x[edge_index[0].long()])
    return out


def gcn_conv_backward_x(g: Tensor, edge_index: Tensor, edge_weight: Optional[Tensor]) -> Tensor:
    """dx[r,h,:] = sum_{e: row_e = r} val_e * g[col_e,h,:]  (transpose SpMM)."""
    val = gcn_edge_values(edge_index, edge_weight, g.shape[0], g.dtype)
    dx = torch.zeros_like(g)
    dx.index_add_(0, edge_index[0].long(), val.view(-1, 1, 1) * g[edge_index[1].long()])
    return dx


# --------------------------------------------------------------------------------------------
# a-4 / a-5  DIFFormerConv.forward (:113-145) and the DIFFormer residual (:197-205)
# --------------------------------------------------------------------------------------------
def _linear(x, w, b):
    return x @ w.T + b


def difformer_conv(sd: Dict[str, Tensor], prefix: str, query_input: Tensor, source_input: Tensor,
                   edge_index, edge_weight, x0, *, num_heads, out_channels, kernel, use_graph,
                   use_weight, graph_weight, use_source) -> Tensor:
    q = _linear(query_input, sd[prefix + "Wq.weight"], sd[prefix + "Wq.bias"]).reshape(-1, num_heads, out_channels)
    k = _linear(source_input, sd[prefix + "Wk.weight"], sd[prefix + "Wk.bias"]).reshape(-1, num_heads, out_channels)
    if use_weight:
        v = _linear(source_input, sd[prefix + "Wv.weight"], sd[prefix + "Wv.bias"]).reshape(-1, num_heads, out_channels)
    else:
        v = source_input.reshape(-1, 1, out_channels)                        # :120
    att = simple_attention(q, k, v) if kernel == "simple" else sigmoid_attention(q, k, v)
    if use_graph:
        g = gcn_conv(v, edge_index, edge_weight)
        fin = (1 - graph_weight) * att + graph_weight * g if graph_weight > 0 else att + g   # :129-134
    else:
        fin = att
    fin = fin.mean(dim=1)                                                    # :137
    if use_source:
        fin = fin + x0                                                       # :139-140
    return fin


def _layer_norm(x, w, b, eps=1e-5):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * w + b


def difformer_forward(sd: Dict[str, Tensor], x: Tensor, edge_index, edge_weight=None, *,
                      hidden_channels, num_layers=2, num_heads=1, kernel="simple", alpha=0.5,
                      use_bn=True, use_residual=True, use_weight=True, use_graph=True,
                      graph_weight=-1, use_source=False) -> Tensor:
    """DIFFormer.forward in eval mode (dropout = identity), difformer.py:184-209."""
    x = _linear(x, sd["fcs.0.weight"], sd["fcs.0.bias"])
    if use_bn:
        x = _layer_norm(x, sd["bns.0.weight"], sd["bns.0.bias"])
    x = torch.relu(x)
    layers = [x]
    for i in range(num_layers):
        y = difformer_conv(sd, f"convs.{i}.", x, x, edge_index, edge_weight, layers[0],
                           num_heads=num_heads, out_channels=hidden_channels, kernel=kernel,
                           use_graph=use_graph, use_weight=use_weight, graph_weight=graph_weight,
                           use_source=use_source)
        if use_residual:
            y = alpha * y + (1 - alpha) * layers[i]                          # :200-201
        if use_bn:
            y = _layer_norm(y, sd[f"bns.{i + 1}.weight"], sd[f"bns.{i + 1}.bias"])
        x = y
        layers.append(x)
    return _linear(x, sd["fcs.1.weight"], sd["fcs.1.bias"])


# --------------------------------------------------------------------------------------------
# a-6  batched-graph 'simple'   physical particle/difformer-v2.py:80-111
# --------------------------------------------------------------------------------------------
def segmented_simple_attention(qs: Tensor, ks: Tensor, vs: Tensor, n_nodes: Tensor) -> Tensor:
    """Per-graph a-1 with N -> n_g (:107-109) but ||Q||_F, ||K||_F over the WHOLE batch (:82-83).
    No padding: plain loop over the graph segments."""
    a, b = torch.linalg.vector_norm(qs), torch.linalg.vector_norm(ks)
    out = torch.empty(qs.shape[0], qs.shape[1], vs.shape[2], dtype=qs.dtype)
    s = 0
    for n in [int(t) for t in n_nodes]:
        q, k, v = qs[s:s + n] / a, ks[s:s + n] / b, vs[s:s + n]
        S = torch.matmul(k.permute(1, 2, 0), v.permute(1, 0, 2))
        num = torch.matmul(q.permute(1, 0, 2), S).permute(1, 0, 2) + v.sum(0).unsqueeze(0)
        den = (q * k.sum(0).unsqueeze(0)).sum(-1) + n
        out[s:s + n] = num / den.unsqueeze(-1)
        s += n
    return out


def segmented_simple_attention_backward(qs, ks, vs, n_nodes, g):
    """Backward of a-6: per-graph a-1b with the global-norm projection applied once at the end."""
    a, b = torch.linalg.vector_norm(qs), torch.linalg.vector_norm(ks)
    qh, kh = qs / a, ks / b
    dqh, dkh, dv = torch.zeros_like(qs), torch.zeros_like(ks), torch.zeros_like(vs)
    s = 0
    for n in [int(t) for t in n_nodes]:
        q, k, v, gg = qh[s:s + n], kh[s:s + n], vs[s:s + n], g[s:s + n]
        S = torch.matmul(k.permute(1, 2, 0), v.permute(1, 0, 2))
        z = k.sum(0)
        den = (q * z.unsqueeze(0)).sum(-1) + n
        out = (torch.matmul(q.permute(1, 0, 2), S).permute(1, 0, 2) + v.sum(0).unsqueeze(0)) / den.unsqueeze(-1)
        dnum = gg / den.unsqueeze(-1)
        dden = -(gg * out).sum(-1) / den
        dqh[s:s + n] = torch.matmul(dnum.permute(1, 0, 2), S.transpose(1, 2)).permute(1, 0, 2) + dden.unsqueeze(-1) * z
        dS = torch.matmul(q.permute(1, 2, 0), dnum.permute(1, 0, 2))
        dz = (q * dden.unsqueeze(-1)).sum(0)
        dkh[s:s + n] = torch.matmul(v.permute(1, 0, 2), dS.transpose(1, 2)).permute(1, 0, 2) + dz
        dv[s:s + n] = torch.matmul(k.permute(1, 0, 2), dS).permute(1, 0, 2) + dnum.sum(0)
        s += n
    dq = (dqh - qh * (qh * dqh).sum()) / a
    dk = (dkh - kh * (kh * dkh).sum()) / b
    return dq, dk, dv


# --------------------------------------------------------------------------------------------
# a-7  batched-graph 'sigmoid'   physical particle/difformer-v2.py:113-135
# --------------------------------------------------------------------------------------------
def segmented_sigmoid_attention(qs: Tensor, ks: Tensor, vs: Tensor, n_nodes: Tensor) -> Tensor:
    """The reference pads every graph to max_node rows (:116-120) and contracts "abcd,ebcd->aebc" (:123): the score couples
    graph a and graph e AT THE SAME PADDED SLOT b, i.e. node b of graph a attends to node b of every graph e (padded slots
    are zero rows: sigmoid(0) = 0.5 in the row sum, zero in the value sum).  Row sums get +1e-9 (:127-128).  Restated slot
    by slot without building the [B,B,M,H] tensors."""
    nn_ = [int(t) for t in n_nodes]
    B, maxn = len(nn_), max(nn_)
    starts = [0]
    for n in nn_:
        starts.append(starts[-1] + n)
    H, D = qs.shape[1], vs.shape[2]
    out = torch.empty(qs.shape[0], H, D, dtype=qs.dtype)
    for b in range(maxn):
        has = [a for a in range(B) if b < nn_[a]]
        idx = torch.tensor([starts[a] + b for a in has], dtype=torch.long)
        qb = torch.zeros(B, H, qs.shape[2], dtype=qs.dtype)
        kb, vb = torch.zeros_like(qb), torch.zeros(B, H, D, dtype=qs.dtype)
        qb[has], kb[has], vb[has] = qs[idx], ks[idx], vs[idx]
        p = torch.sigmoid(torch.matmul(qb.permute(1, 0, 2), kb.permute(1, 2, 0)))     # [H, B(a), B(e)]
        att = p / (p.sum(-1, keepdim=True) + 1e-9)
        ob = torch.matmul(att, vb.permute(1, 0, 2)).permute(1, 0, 2)                   # [B, H, D]
        out[idx] = ob[has]
    return out


def difformer_v2_forward(sd: Dict[str, Tensor], x: Tensor, edge_index, n_nodes, *, hidden_channels,
                         num_layers=2, alpha=0.5, use_bn=True, use_residual=True, use_graph=True,
                         graph_weight=-1) -> Tensor:
    """DIFFormer_v2.forward in eval mode, kernel='simple', use_weight=True (TransConv.forward
    requires it: `value` is only bound under use_weight, difformer-v2.py:149-150).  H is always 1
    (:177).  ReLU after every layer (:216), difformer-v2.py:196-223."""
    x = _linear(x, sd["fcs.0.weight"], sd["fcs.0.bias"])
    if use_bn:
        x = _layer_norm(x, sd["bns.0.weight"], sd["bns.0.bias"])
    x = torch.relu(x)
    layers = [x]
    for i in range(num_layers):
        p = f"convs.{i}."
        q = _linear(x, sd[p + "Wq.weight"], sd[p + "Wq.bias"]).reshape(-1, 1, hidden_channels)
        k = _linear(x, sd[p + "Wk.weight"], sd[p + "Wk.bias"]).reshape(-1, 1, hidden_channels)
        v = _linear(x, sd[p + "Wv.weight"], sd[p + "Wv.bias"]).reshape(-1, 1, hidden_channels)
        att = segmented_simple_attention(q, k, v, n_nodes)
        if use_graph:
            g = gcn_conv(v, edge_index, None)
            fin = (1 - graph_weight) * att + graph_weight * g if graph_weight > 0 else att + g
        else:
            fin = att
        y = fin.mean(dim=1)
        if use_residual:
            y = alpha * y + (1 - alpha) * layers[i]
        if use_bn:
            y = _layer_norm(y, sd[f"bns.{i + 1}.weight"], sd[f"bns.{i + 1}.bias"])
        x = torch.relu(y)
        layers.append(x)
    return _linear(x, sd["fcs.1.weight"], sd["fcs.1.bias"])


# --------------------------------------------------------------------------------------------
# helpers shared by tests / bench (synthetic inputs, SURVEY.md section 8d)
# --------------------------------------------------------------------------------------------
def synthetic_qkv(n: int, h: int, d: int, seed: int = 123, hv: Optional[int] = None,
                  adversarial: bool = False, dtype=torch.float32):
    """Seeded N(0,1) Q,K,V.  `adversarial`: Q,K get mean 0.5 and V is column-centred up to a small
    0.02 offset, which exercises sum_k and defeats the mean-collapse of 'simple' (SURVEY.md
    section 8a warning).  The offset keeps u = sum(V) well-conditioned: with *exactly* centred V the
    reference's own fp32 output is cancellation noise (it differs from fp64 by > 1e-3)."""
    gen = torch.Generator().manual_seed(seed)
    hv = h if hv is None else hv
    q = torch.randn(n, h, d, generator=gen, dtype=dtype)
    k = torch.randn(n, h, d, generator=gen, dtype=dtype)
    v = torch.randn(n, hv, d, generator=gen, dtype=dtype)
    if adversarial:
        q, k = q + 0.5, k + 0.5
        v = v - v.mean(0, keepdim=True) + 0.02
    return q, k, v


def synthetic_graph(n: int, n_pairs: int, seed: int = 123, self_loops: bool = True) -> Tensor:
    """Random undirected pairs -> both directions (+ self loops), like main.py:72-79 produces."""
    gen = torch.Generator().manual_seed(seed)
    a = torch.randint(0, n, (n_pairs,), generator=gen)
    b = torch.randint(0, n, (n_pairs,), generator=gen)
    keep = a != b
    a, b = a[keep], b[keep]
    row, col = torch.cat([a, b]), torch.cat([b, a])
    if self_loops:
        loop = torch.arange(n)
        row, col = torch.cat([row, loop]), torch.cat([col, loop])
    return torch.stack([row, col]).long()


def rel_err(x: Tensor, ref: Tensor) -> float:
    """Norm-wise relative error ||x-ref||/||ref|| evaluated in fp64 (on the GPU when either side lives there: the
    full-size bench checks compare multi-GB tensors)."""
    dev = x.device if x.is_cuda else ref.device
    x, ref = x.detach().to(dev, torch.float64), ref.detach().to(dev, torch.float64)
    den = float(torch.linalg.vector_norm(ref))
    return float(torch.linalg.vector_norm(x - ref)) / (den if den > 0 else 1.0)


def projected_operands(G: Tensor, s: Tensor, n_total: float, Wq: Tensor, bq: Tensor, Wk: Tensor, bk: Tensor,
                       Wv: Optional[Tensor], bv: Optional[Tensor], H: int):
    """The pass-2 operands of 'simple' attention when Q = x Wq^T + bq, K = x Wk^T + bk, V = x Wv^T + bv (difformer.py:115-120) are
    never formed: everything full_attention_conv (difformer.py:18-39) reduces over the rows follows from G = X^T X and s = X^T 1.
    fp64 torch restatement of difformer_b200/csrc/project.cu (test infrastructure).  Weights in nn.Linear layout [H*C, C] / [H*C];
    Wv = None: V_h = x.  Returns (vpartials [H*C*C + 2*H*C + 2], nvec [H], wbar [C, C], bbar [C]) in fp64:
        vpartials = [Wq_h^T S_h | Wq_h^T z_h | u_h + c bq_h^T S_h | sum q^2 | sum k^2],  nvec[h] = n + c bq_h . z_h."""
    C = G.shape[0]
    G, s = G.double(), s.double()
    Wq, bq = Wq.double().view(H, C, C), bq.double().view(H, C)
    Wk, bk = Wk.double().view(H, C, C), bk.double().view(H, C)
    if Wv is not None:
        Wv, bv = Wv.double().view(H, C, C), bv.double().view(H, C)
    else:
        Wv = torch.eye(C, dtype=torch.float64).expand(H, C, C)
        bv = torch.zeros(H, C, dtype=torch.float64)
    n = float(n_total)
    ks, vs, qs = Wk @ s, Wv @ s, Wq @ s
    S = Wk @ G @ Wv.transpose(1, 2) + ks.unsqueeze(2) * bv.unsqueeze(1) + bk.unsqueeze(2) * vs.unsqueeze(1) \
        + n * bk.unsqueeze(2) * bv.unsqueeze(1)
    z = ks + n * bk
    u = vs + n * bv
    sk = ((Wk @ G) * Wk).sum() + 2.0 * (bk * ks).sum() + n * (bk * bk).sum()
    sq = ((Wq @ G) * Wq).sum() + 2.0 * (bq * qs).sum() + n * (bq * bq).sum()
    c = 1.0 / torch.sqrt(sq * sk)
    A = Wq.transpose(1, 2) @ S
    a = (bq.unsqueeze(1) @ S).squeeze(1)
    w = (Wq.transpose(1, 2) @ z.unsqueeze(2)).squeeze(2)
    beta = (bq * z).sum(1)
    vpart = torch.cat([A.reshape(-1), w.reshape(-1), (u + c * a).reshape(-1), sq.reshape(1), sk.reshape(1)])
    return vpart, n + c * beta, Wv.mean(0), bv.mean(0)


def segmented_tile_plan(n_nodes: Tensor, max_nodes: Optional[int] = None):
    """Restatement of the device-side plan of the tensor-core batched-graph kernels (difformer_b200/csrc/segmented_sm100.cu,
    seg_plan_kernel): whole graphs packed into tiles of at most 128 rows without a sequential pass.  Tile b holds the graphs whose FIRST
    row lies in [b S, (b + 1) S), S = 129 - max_nodes.  Returns (tile_row0 [ntiles + 1], row_range [N, 2]) as int64 tensors."""
    nn_ = n_nodes.to(torch.int64)
    ptr = torch.zeros(nn_.numel() + 1, dtype=torch.int64)
    ptr[1:] = torch.cumsum(nn_, 0)
    N = int(ptr[-1])
    mx = int(nn_.max()) if max_nodes is None else int(max_nodes)
    S = 129 - mx
    ntiles = (N + S - 1) // S
    tile_row0 = torch.full((ntiles + 1,), -1, dtype=torch.int64)
    row_range = torch.zeros((N, 2), dtype=torch.int64)
    prev_bucket = -1
    for g in range(nn_.numel()):
        s_, e_ = int(ptr[g]), int(ptr[g + 1])
        if e_ <= s_:
            continue                                   # an empty graph owns no rows
        row_range[s_:e_, 0] = s_
        row_range[s_:e_, 1] = e_
        b = s_ // S
        tile_row0[prev_bucket + 1:b + 1] = s_          # this graph opens bucket b (and any empty buckets before it)
        prev_bucket = b
        if e_ == N:
            tile_row0[b + 1:] = N
    return tile_row0, row_range

