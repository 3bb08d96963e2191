"""GPU: round-2 parity tests.

  * K7 losses (log_softmax + NLL, GradientTailLoss) against torch, forward and backward, fp32 and bf16 logits;
  * any multi_hop_max_dist in 1..32 (the reference's default is 5): K1 + K2 against the oracle;
  * a reference-collated dense batch is accepted by Graphormer.forward;
  * the evaluation steps run the fused K5 head: ranks / top-k equal those of the full logits, metrics equal the reference's;
  * the padding row of the time table receives no gradient (nn.Embedding(padding_idx=0));
  * K5 against an independent fp32 GEMM on a well-separated case;
  * the canonical model (6 layers, ffn 1024) on BASELINE-shaped batches — configs[1] (128-node graphs, 60 000 POIs) and
    configs[3] (<= 256-node graphs, 3 679 POIs) — forward, loss and EVERY parameter gradient against the oracle;
  * `entry.cli_main` with the reference's README flags: 3 training steps, then --test.
"""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import model_oracle as mo

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


# ------------------------------------------------------------------------------------------------------- K7
@pytest.mark.parametrize("B,V,dtype", [(256, 60001, torch.float32), (37, 3680, torch.float32), (64, 5000, torch.bfloat16),
                                       (5, 98, torch.float32)])
def test_k7_log_softmax_nll(lib_built, B, V, dtype):
    from mobgt_b200 import ops
    g = torch.Generator().manual_seed(B + V)
    x = (torch.randn(B, V, generator=g) * 3).to(dtype)
    t = torch.randint(0, V, (B,), generator=g)
    t[::5] = 0                                                     # ignore_index rows
    xr = x.float().clone().requires_grad_(True)
    ref = F.nll_loss(F.log_softmax(xr, dim=1), t, ignore_index=0)
    (ref * 1.7).backward()
    xg = x.cuda().requires_grad_(True)
    got = ops.log_softmax_nll_loss(xg, t.cuda(), ignore_index=0)
    (got * 1.7).backward()
    tol = 1e-5 if dtype == torch.float32 else 2e-2
    assert abs(got.item() - ref.item()) <= tol * abs(ref.item()), (got.item(), ref.item())
    gr = xr.grad
    err = (xg.grad.float().cpu() - gr).abs().max().item()
    assert err <= tol * gr.abs().max().item() + 1e-9, err
    assert (xg.grad[::5] == 0).all()                               # ignored rows: exact zeros
    # bitwise reproducible
    got2 = ops.log_softmax_nll_loss(xg.detach(), t.cuda(), ignore_index=0)
    assert got2.item() == got.item()


@pytest.mark.parametrize("B,V,alpha,dtype", [(256, 3679, 0.2, torch.float32), (256, 300, 0.1, torch.float32), (16, 60000, 0.2, torch.float32),
                                             (32, 1000, 0.2, torch.bfloat16)])
def test_k7_gradient_tail_loss(lib_built, B, V, alpha, dtype):
    from mobgt_b200 import ops
    g = torch.Generator().manual_seed(B * 7 + V)
    x = (torch.randn(B, V, generator=g) * 2).to(dtype)
    t = torch.randint(0, V, (B + 3,), generator=g)                 # longer than the batch: `targets[:len(inputs)]` (:547)
    xr = x.float().clone().requires_grad_(True)
    ref = mo.gradient_tail_loss(xr, t, alpha)
    (ref * 0.5).backward()
    xg = x.cuda().requires_grad_(True)
    got = ops.gradient_tail_loss(xg, t.cuda(), alpha)
    (got * 0.5).backward()
    tol = 1e-5 if dtype == torch.float32 else 2e-2
    assert abs(got.item() - ref.item()) <= tol * abs(ref.item()), (got.item(), ref.item())
    gr = xr.grad
    assert (xg.grad.float().cpu() - gr).abs().max().item() <= tol * gr.abs().max().item() + 1e-12


# ------------------------------------------------------------------------------------------------------- K10
@pytest.mark.parametrize("M,N,K,mode", [(1000, 640, 192, 0), (33024, 1024, 192, 1), (4100, 256, 1024, 0), (130, 256, 192, 1),
                                        (5, 128, 192, 0), (3000, 1024, 192, 2), (33024, 1024, 192, 2), (77, 256, 192, 2),
                                        (640, 128, 64, 0), (300, 128, 576, 0)])
def test_k10_gemm_epilogues(lib_built, M, N, K, mode):
    """tcgen05 GEMM with fused epilogues against torch fp32 on the same bf16 operands: mode 0 (+ bias), mode 1 (+ bias, GELU),
    mode 2 (FFN backward: (a w^T) o gelu'(a2 w2^T + bias) and its column sums).  bf16 output: 2^-8 relative.  Both GELU forms
    of the epilogue — the default erf form and the optional tanh form on MUFU.TANH — are compared with torch's exact nn.GELU."""
    from mobgt_b200 import _C
    try:
        for exact in ((1, 0) if mode else (1,)):
            _C.call("mobgt_gemm_exact_gelu", exact)
            _k10_case(M, N, K, mode)
    finally:
        _C.call("mobgt_gemm_exact_gelu", 1)


def _k10_case(M, N, K, mode):
    from mobgt_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M + N + K + mode)
    a = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).to(torch.bfloat16)
    bias = torch.randn(N, device="cuda", generator=g) * 0.5
    if mode < 2:
        got = ops.gemm_bf16(a, w, bias, mode=mode)
        ref = a.float() @ w.float().t() + bias
        if mode == 1:
            ref = F.gelu(ref)
        err = (got.float() - ref).abs().max().item()
        assert err <= 1e-2 * max(1.0, ref.abs().max().item()), err
        assert torch.equal(got, ops.gemm_bf16(a, w, bias, mode=mode))                  # bitwise reproducible
        # the same result through a strided A (a column slice of a wider matrix)
        wide = torch.cat([a, a], 1)
        assert torch.equal(got, ops.gemm_bf16(wide[:, K:], w, bias, mode=mode))
        return
    K2 = 192
    a2 = torch.randn(M, K2, device="cuda", generator=g).to(torch.bfloat16)
    w2 = (torch.randn(N, K2, device="cuda", generator=g) / K2 ** 0.5).to(torch.bfloat16)
    got, cs = ops.gemm_bf16(a, w, bias, mode=2, a2=a2, w2=w2, want_colsum=True)
    h = (a2.float() @ w2.float().t() + bias).requires_grad_(True)
    up = a.float() @ w.float().t()
    F.gelu(h).backward(up)
    ref = h.grad
    err = (got.float() - ref).abs().max().item()
    assert err <= 1e-2 * max(1.0, ref.abs().max().item()), err
    cref = got.float().sum(0)                                                         # column sums of what was stored
    assert (cs - cref).abs().max().item() <= 1e-3 * max(1.0, cref.abs().max().item())


# ------------------------------------------------------------------------------------------------------- K9
def test_k9_flat_adamw_matches_torch(lib_built):
    """optim.FlatAdamW (one kernel over flat buffers) against torch.optim.AdamW on the same parameters and gradients, five steps
    with a changing learning rate; parameters stay views of the flat buffer and a bf16 working copy notices the update."""
    from mobgt_b200 import ops
    from mobgt_b200.optim import FlatAdamW
    torch.manual_seed(0)
    shapes = [(60001, 320), (320,), (192, 1024), (7,), (1, 8), (128 * 64, 1)]
    ours = [torch.nn.Parameter(torch.randn(s, device="cuda")) for s in shapes]
    ref = [torch.nn.Parameter(p.detach().clone()) for p in ours]
    o1 = FlatAdamW(ours, lr=2e-4, weight_decay=0.01)
    o2 = torch.optim.AdamW(ref, lr=2e-4, weight_decay=0.01)
    lin = torch.nn.Linear(1024, 192).cuda()
    w16 = ops.Bf16Weights()
    holder = torch.nn.Linear(1024, 192).cuda()
    holder.weight, holder.bias = ours[2], torch.nn.Parameter(torch.zeros(192, device="cuda"))
    w16.register("k", [holder])
    w16.refresh()
    for step in range(5):
        lr = 2e-4 * (step + 1) / 5
        for grp in o1.param_groups + o2.param_groups:
            grp["lr"] = lr
        for a, b in zip(ours, ref):
            gnew = torch.randn_like(a) * (0.1 + step)
            a.grad.copy_(gnew)                      # gradients are views of the flat buffer: written in place
            b.grad = gnew.clone()
        o1.step()
        o2.step()
    for a, b in zip(ours, ref):
        assert a.data_ptr() >= o1.flat_param.data_ptr() and a.data_ptr() < o1.flat_param.data_ptr() + o1.n * 4
        assert a.data_ptr() % 16 == 0 and a.grad.data_ptr() % 16 == 0          # kernels read parameters with 128-bit loads
        assert (a.detach() - b.detach()).abs().max().item() <= 2e-6 * max(1.0, b.abs().max().item())
    w16.refresh()
    assert torch.equal(w16.get("k")[0], ours[2].detach().to(torch.bfloat16))
    del lin


# ------------------------------------------------------------------------------------------------------- K8
@pytest.mark.parametrize("n,D,density", [(300, 16, 0.2), (3679, 64, 0.01), (60000, 16, 0.0005), (5000, 128, 0.004), (253, 32, 0.2)])
def test_k8_spmm_csr_forward_backward(lib_built, n, D, density):
    """Y = LeakyReLU(A @ S + b) and its gradients against torch on the dense matrix (fp32; sums in a different order: 1e-5)."""
    from mobgt_b200 import ops
    from mobgt_b200.model import _csr_transpose
    rng = np.random.default_rng(n + D)
    nnz_row = np.maximum(1, rng.poisson(density * n, size=n))
    nnz_row[rng.integers(0, n, 3)] = 0                                           # empty rows
    crow = np.zeros(n + 1, np.int64)
    np.cumsum(nnz_row, out=crow[1:])
    col = np.concatenate([np.sort(rng.choice(n, size=k, replace=False)) for k in nnz_row]).astype(np.int64)
    val = rng.random(len(col)).astype(np.float32)
    A = tuple(torch.from_numpy(np.ascontiguousarray(a, dt)).cuda() for a, dt in zip((crow, col, val), (np.int32, np.int32, np.float32)))
    At = tuple(torch.from_numpy(np.ascontiguousarray(a, dt)).cuda() for a, dt in zip(_csr_transpose((crow, col, val), n), (np.int32, np.int32, np.float32)))
    g = torch.Generator().manual_seed(1)
    S = torch.randn(n, D, generator=g)
    b = torch.randn(D, generator=g)
    dY = torch.randn(n, D, generator=g)
    dense = torch.sparse_csr_tensor(torch.from_numpy(crow), torch.from_numpy(col), torch.from_numpy(val), size=(n, n)).to_dense() \
        if n <= 6000 else None
    for slope in (None, 0.2):
        Sg, bg = S.cuda().requires_grad_(True), b.cuda().requires_grad_(True)
        Y = ops.spmm(A, At, Sg, bg, slope)
        (Y * dY.cuda()).sum().backward()
        Sr, br = S.clone().requires_grad_(True), b.clone().requires_grad_(True)
        if dense is not None:
            Z = dense @ Sr + br
        else:
            Z = torch.sparse.mm(torch.sparse_csr_tensor(torch.from_numpy(crow), torch.from_numpy(col), torch.from_numpy(val), size=(n, n)), Sr) + br
        Yr = F.leaky_relu(Z, slope) if slope is not None else Z
        (Yr * dY).sum().backward()
        for got, ref, name in ((Y, Yr, "Y"), (Sg.grad, Sr.grad, "dS"), (bg.grad, br.grad, "db")):
            err = (got.detach().cpu() - ref.detach()).abs().max().item()
            assert err <= 2e-5 * max(1.0, ref.abs().max().item()), (name, slope, err)
    # no bias, bitwise reproducible
    Y1, Y2 = ops.spmm_csr_raw(A, S.cuda()), ops.spmm_csr_raw(A, S.cuda())
    assert torch.equal(Y1, Y2)


# ------------------------------------------------------------------------------------------------------- K3 bwd, single-box variant
@pytest.mark.parametrize("sizes", [(128, 128, 5, 128), (127, 100, 1, 64, 33, 17, 128), (12, 3, 7, 1, 9)])
def test_attention_bwd_single_box_variant(lib_built, sizes):
    """mobgt_attn_bwd in mode 2 (per-layer bf16 dS plane) on batches whose graphs all have <= 128 nodes takes the two-CTA-per-SM
    single-box kernel (csrc/k3_attn_bwd.cu: k3_attn_bwd1_kernel).  dq / dk / dv and the dS plane against torch autograd with the
    same dropout mask, and against the general kernel (mode 0, fp32 dS)."""
    from mobgt_b200 import collator, ops, synth
    from test_k2_k3_k4 import tables, torch_attention_diff
    w = synth.make_world("c1", seed=1)
    items = []
    for k, n in enumerate(sizes):
        items += synth.make_items(w, 1, 512, seed=70 + k, n_fixed=n, start=k)
    b = collator.collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=1024, world=w)
    assert b.N <= 128
    B = len(items)
    R, Pp, E, W, t = tables(seed=4)
    cu = [x.cuda().contiguous() for x in (R, Pp, E, W.view(-1), t.view(-1))]
    bias = ops.bias_fwd_raw(b, *cu, out_dtype=torch.bfloat16)
    ntok = int(b.tok_pos.numel())
    gen = torch.Generator().manual_seed(13)
    qkv = (torch.randn(ntok, 3 * 192, generator=gen) * 1.2).to(torch.bfloat16)
    dout = torch.randn(ntok, 192, generator=gen).to(torch.bfloat16)
    tok_off = b.tok_off.cpu().numpy()
    for p, seed in ((0.0, 0), (0.1, 0x0123456789ABCDEF)):
        out, lse = ops.attn_fwd_raw(qkv.cuda(), bias, b, drop_p=p, seed=seed)
        plane = torch.full(bias.shape, float("nan"), dtype=torch.bfloat16, device="cuda")
        dqkv = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, plane, 2, drop_p=p, seed=seed)        # single-box kernel
        db32 = torch.full(bias.shape, float("nan"), dtype=torch.float32, device="cuda")
        dqkv0 = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, db32, 0, drop_p=p, seed=seed)        # general kernel
        torch.cuda.synchronize()
        q32 = qkv.float().requires_grad_(True)
        b32 = bias.float().cpu().requires_grad_(True)
        ref, _ = torch_attention_diff(q32, b32, tok_off, drop=(p, seed) if p > 0 else None)
        (ref * dout.float()).sum().backward()
        gq = q32.grad
        err = (dqkv.float().cpu() - gq).abs().max().item()
        assert err <= 2e-2 * max(1.0, gq.abs().max().item()), f"p={p}: dqkv max err {err}"
        assert (dqkv.float() - dqkv0.float()).abs().max().item() <= 1e-2 * max(1.0, gq.abs().max().item())
        for g in range(B):
            Tg = int(tok_off[g + 1] - tok_off[g])
            gb = b32.grad[g, :, :Tg, :Tg]
            got = plane[g, :, :Tg, :Tg].float().cpu()
            assert torch.isfinite(got).all(), (p, g)
            assert (got - gb).abs().max().item() <= 2e-2 * max(1.0, gb.abs().max().item()), (p, g)
            assert (got - db32[g, :, :Tg, :Tg].cpu()).abs().max().item() <= 1e-2 * max(1.0, gb.abs().max().item()), (p, g)
    # bitwise reproducible
    plane2 = torch.empty_like(plane)
    dq2 = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, plane2, 2, drop_p=p, seed=seed)
    assert torch.equal(dq2, dqkv)


# ------------------------------------------------------------------------------------------------------- K3: persistent CTAs, size classes
@pytest.mark.parametrize("p_drop", [0.0, 0.1])
def test_attention_many_items_all_size_classes(lib_built, p_drop):
    """More (graph, head) work items than the forward kernel has persistent CTAs (2 x 148), with every size class in one
    batch: graphs of <= 16 tokens (SIMT kernels, csrc/k3_attn_small.cu), single-box graphs, the 128 m + 1 single-token tails
    (T = 129, 257), two- and three-box graphs.  Forward, lse and the backward (general kernel, fp32 dS, mode 0 then mode 1
    accumulating on top) against torch autograd with the same dropout mask: the barrier phases of a persistent CTA run on across
    items of different shapes, and the tensor-core and SIMT kernels split the batch on the device."""
    from mobgt_b200 import collator, ops, synth
    from test_k2_k3_k4 import tables, torch_attention_diff
    w = synth.make_world("c1", seed=1)
    sizes = [128, 5, 100, 256, 1, 15, 130, 16, 3, 128, 64, 300, 2, 33, 17, 127, 8, 200, 12, 256, 4, 90, 128, 6] + [3 + (i * 7) % 40 for i in range(24)]
    items = []
    for k, n in enumerate(sizes):
        items += synth.make_items(w, 1, 512, seed=170 + k, n_fixed=n, start=k)
    b = collator.collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=1024, world=w)
    B = len(items)
    assert B * 8 > 2 * 148
    R, Pp, E, W, t = tables(seed=4)
    cu = [x.cuda().contiguous() for x in (R, Pp, E, W.view(-1), t.view(-1))]
    bias = ops.bias_fwd_raw(b, *cu, out_dtype=torch.bfloat16)
    ntok = int(b.tok_pos.numel())
    gen = torch.Generator().manual_seed(21)
    qkv = (torch.randn(ntok, 3 * 192, generator=gen) * 1.2).to(torch.bfloat16)
    dout = torch.randn(ntok, 192, generator=gen).to(torch.bfloat16)
    tok_off = b.tok_off.cpu().numpy()
    seed = 0x0F1E2D3C4B5A6978
    out, lse = ops.attn_fwd_raw(qkv.cuda(), bias, b, drop_p=p_drop, seed=seed)
    db32 = torch.full(bias.shape, float("nan"), dtype=torch.float32, device="cuda")
    dqkv = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, db32, 0, drop_p=p_drop, seed=seed)
    torch.cuda.synchronize()
    q32 = qkv.float().requires_grad_(True)
    b32 = bias.float().cpu().requires_grad_(True)
    ref, ref_lse = torch_attention_diff(q32, b32, tok_off, drop=(p_drop, seed) if p_drop > 0 else None)
    (ref * dout.float()).sum().backward()
    assert torch.isfinite(out.float()).all() and torch.isfinite(lse).all()
    assert (out.float().cpu() - ref.detach()).abs().max().item() <= 2e-2 * max(1.0, ref.abs().max().item())
    with torch.no_grad():                   # lse [ntok, H] = logsumexp of the biased scores (before the dropout mask)
        for g in range(B):
            a, e = int(tok_off[g]), int(tok_off[g + 1])
            T = e - a
            q = q32[a:e, :192].view(T, 8, 24).transpose(0, 1)
            k = q32[a:e, 192:384].view(T, 8, 24).transpose(0, 1)
            sc = (q * 24 ** -0.5) @ k.transpose(1, 2) + b32[g, :, :T, :T]
            want = torch.logsumexp(sc, -1).transpose(0, 1)
            assert (lse[a:e].cpu() - want).abs().max().item() <= 2e-2, g
    gq = q32.grad
    assert (dqkv.float().cpu() - gq).abs().max().item() <= 2e-2 * max(1.0, gq.abs().max().item())
    acc = db32.clone()
    for g in range(B):                      # unwritten cells of the fp32 plane are not numbers: accumulate on the live corner only
        Tg = int(tok_off[g + 1] - tok_off[g])
        gb = b32.grad[g, :, :Tg, :Tg]
        got = db32[g, :, :Tg, :Tg].cpu()
        assert torch.isfinite(got).all(), g
        assert (got - gb).abs().max().item() <= 2e-2 * max(1.0, gb.abs().max().item()), (g, Tg)
    acc = torch.nan_to_num(acc, nan=0.0)
    ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, acc, 1, drop_p=p_drop, seed=seed)     # mode 1: += dS
    for g in range(B):
        Tg = int(tok_off[g + 1] - tok_off[g])
        gb = b32.grad[g, :, :Tg, :Tg]
        assert (acc[g, :, :Tg, :Tg].cpu() - 2 * gb).abs().max().item() <= 4e-2 * max(1.0, gb.abs().max().item()), (g, Tg)


# ------------------------------------------------------------------------------------------------------- multi_hop_max_dist
def _tables(H=8, bins=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    R = torch.randn(512, H, generator=g) * 0.3
    Pp = torch.randn(bins, H, generator=g) * 0.3
    E = torch.randn(128, H, generator=g) * 0.3
    W = torch.randn(128 * H * H, 1, generator=g) * 0.3
    t = torch.randn(1, H, generator=g) * 0.3
    R[0] = 0
    Pp[0] = 0
    E[0] = 0
    return R, Pp, E, W, t


def _oracle_bias(ob, R, Pp, E, W, t, dk, H=8):
    m = mo.Graphormer.__new__(mo.Graphormer)
    torch.nn.Module.__init__(m)
    m.num_heads, m.multi_hop_max_dist = H, dk
    m.rel_pos_encoder = torch.nn.Embedding.from_pretrained(R.clone(), freeze=False, padding_idx=0)
    m.poi_pos_encoder = torch.nn.Embedding.from_pretrained(Pp.clone(), freeze=False, padding_idx=0)
    m.edge_encoder = torch.nn.Embedding.from_pretrained(E.clone(), freeze=False, padding_idx=0)
    m.edge_dis_encoder = torch.nn.Embedding.from_pretrained(W.clone(), freeze=False)
    m.graph_token_virtual_distance = torch.nn.Embedding.from_pretrained(t.clone(), freeze=False)
    return m, m.attn_bias_build(ob, "fp32")


@pytest.mark.parametrize("dk", [5, 1, 7, 13, 32])
def test_any_multi_hop_max_dist(lib_built, dk):
    """The reference's default --multi_hop_max_dist is 5 (entry.py / data.py:204).  K1 walks dk hops into rows of
    hop_stride(dk) bytes; K2 clamps the mean at dk.  Collated fields bit-exact, bias fwd 1e-5 (fp32), bias bwd vs autograd."""
    from mobgt_b200 import collator, ops, synth
    w = synth.make_world("c1", seed=1)
    items = synth.make_items(w, 6, 50, seed=dk)
    ob = mo.collate([mo.preprocess_item(it, hop_cap=32) for it in items], w, multi_hop_max_dist=dk, rel_pos_max=1024)
    b = collator.collator_toyota(items, max_node=512, multi_hop_max_dist=dk, rel_pos_max=1024, world=w)
    assert b.dk == dk and b.hops % 4 == 0
    assert torch.equal(b.rel_pos.cpu(), ob.rel_pos)
    assert b.edge_input.shape == ob.edge_input.shape and torch.equal(b.edge_input.cpu(), ob.edge_input)
    R, Pp, E, W, t = _tables(seed=dk)
    m, ref = _oracle_bias(ob, R, Pp, E, W, t, dk)
    cu = [x.cuda().contiguous() for x in (R, Pp, E, W.view(-1), t.view(-1))]
    out32 = ops.bias_fwd_raw(b, *cu, out_dtype=torch.float32).cpu()
    B, H, T = ref.shape[0], 8, b.N + 1
    for g in range(B):
        Tg = int(b.n_host[g]) + 1
        assert torch.allclose(out32[g, :, :Tg, :Tg], ref[g, :, :Tg, :Tg].detach(), rtol=1e-5, atol=1e-6), (dk, g)
    Tp = ops.bias_pitch(T)
    gen = torch.Generator().manual_seed(5)
    dB = torch.zeros(B, H, T, Tp)
    for g in range(B):
        Tg = int(b.n_host[g]) + 1
        dB[g, :, :Tg, :Tg] = torch.randn(H, Tg, Tg, generator=gen)
    finite = torch.where(torch.isfinite(ref), ref, torch.zeros_like(ref))
    (finite * dB[..., :T]).sum().backward()
    dR, dP, dE, dW, dt = ops.bias_bwd_raw(b, dB.cuda(), E.cuda().contiguous(), W.view(-1).cuda().contiguous(), Pp.shape[0])
    for got, exp, name in ((dR, m.rel_pos_encoder.weight.grad, "dR"), (dP, m.poi_pos_encoder.weight.grad, "dP"),
                           (dE, m.edge_encoder.weight.grad, "dE"), (dW.view(-1, 1), m.edge_dis_encoder.weight.grad, "dW"),
                           (dt.view(1, -1), m.graph_token_virtual_distance.weight.grad, "dt")):
        scale = exp.abs().max().item() + 1e-6
        assert (got.cpu() - exp).abs().max().item() <= 2e-5 * scale + 1e-5, (dk, name)


# ------------------------------------------------------------------------------------------------------- model level
def _pair(dataset_name, cfg, items_spec, n_layers=2, ffn=256, seed=1, dk=20, scale_tables=True, **model_kw):
    """oracle model + product model with the same weights, oracle batch + product batch of the same items."""
    from mobgt_b200 import collator, model, synth
    w = synth.make_world(cfg, seed=seed, dataset_name=dataset_name)
    items = []
    for n_fixed, cnt, cap, sd in items_spec:
        items += synth.make_items(w, cnt, cap, seed=sd, n_fixed=n_fixed, start=len(items))
    hp = dict(n_layers=n_layers, num_heads=8, hidden_dim=128, dropout_rate=0.0, intput_dropout_rate=0.0, weight_decay=0.01,
              ffn_dim=ffn, warmup_updates=10, tot_updates=100, peak_lr=2e-4, end_lr=1e-9, edge_type="multi_hop",
              multi_hop_max_dist=dk, attention_dropout_rate=0.0)
    torch.manual_seed(seed)
    om = mo.Graphormer(w, n_layers=n_layers, ffn_dim=ffn, dataset_name=dataset_name, multi_hop_max_dist=dk).eval()
    if scale_tables:
        with torch.no_grad():
            for emb in (om.edge_encoder, om.rel_pos_encoder, om.poi_pos_encoder):
                emb.weight.mul_(0.3)
                emb.weight[0].zero_()
            om.edge_dis_encoder.weight.mul_(0.3)
    pm = model.Graphormer(dataset_name=dataset_name, world=w, **hp, **model_kw).cuda().eval()
    missing, _ = pm.load_state_dict(om.state_dict(), strict=False)
    assert not missing, missing
    ob = mo.collate([mo.preprocess_item(it, hop_cap=max(20, dk)) for it in items], w, multi_hop_max_dist=dk, rel_pos_max=1024)
    pb = collator.collator_toyota(items, max_node=512, multi_hop_max_dist=dk, rel_pos_max=1024, world=w)
    return w, items, om, pm, ob, pb


def test_forward_accepts_reference_collated_dense_batch(lib_built):
    """A dense Batch1 as the REFERENCE's collator builds it (padded int64 / fp32 CPU tensors, here the oracle's pinned
    restatement) goes straight into Graphormer.forward; logits equal those of the packed batch of the same items bit for bit."""
    w, items, om, pm, ob, pb = _pair("gowalla_nevda", "tiny", [(None, 6, 12, 4)], dk=5)
    with torch.no_grad():
        a = pm(pb)
        d = pm(ob)
        ref = om(ob)
    assert torch.equal(a[0], d[0]) and torch.equal(a[1], d[1])
    assert (a[0].float().cpu() - ref[0]).abs().max().item() <= 2e-2 * max(1.0, ref[0].abs().max().item())


@pytest.mark.parametrize("dataset_name", ["toyotagraph", "gowalla_nevda", "foursquaregraph"])
def test_eval_steps_run_the_fused_head(lib_built, dataset_name):
    """validation_step / test_step (model_fqandtoyo.py:1484-1544) through K5: top-20 ids and target ranks equal those of the
    logits the same step returns on request, y_true follows the reference's per-dataset rule, and test_epoch_end prints the
    metrics the reference's get_acc / MRR_metric give on those logits."""
    from mobgt_b200 import _C
    w, items, om, pm, ob, pb = _pair(dataset_name, "c1", [(None, 24, 30, 9)])
    n0 = _C.launch_count()
    with torch.no_grad():
        out = pm.test_step(pb, full_logits=True)
        fast = pm.test_step(pb)
    assert "y_pred" not in fast and _C.launch_count() > n0
    y_true = pb.y if dataset_name == "toyotagraph" else pb.y - 1
    assert torch.equal(out["y_true"], y_true)
    # the fused head computes bf16 x bf16 -> fp32; build the same logits independently
    z, _ = pm.features(pb)
    lg = z.detach().to(torch.bfloat16).float() @ pm.out_proj.weight.detach().to(torch.bfloat16).float().t() + pm.out_proj.bias.detach()
    st = lg.gather(1, y_true.view(-1, 1))
    idx = torch.arange(lg.shape[1], device=lg.device).view(1, -1)
    rank = (lg > st).sum(1) + ((lg == st) & (idx < y_true.view(-1, 1))).sum(1)
    near = ((lg - st).abs() < 1e-5 * lg.abs().max()).sum(1) > 1                   # another logit within rounding of the target's
    assert ((out["rank"].long() == rank) | near).all()
    assert torch.equal(fast["rank"], out["rank"]) and torch.equal(fast["idx"], out["idx"])
    tv, ti = lg.topk(21, dim=1)
    decisive = ((tv[:, :-1] - tv[:, 1:]).abs() > 1e-5 * tv.abs().max()).all(1)
    assert ((out["idx"].long() == ti[:, :20]).all(1) | ~decisive).all()
    # metrics: product epoch end == the reference's functions on the bf16-operand logits
    res = pm.test_epoch_end([fast], quiet=True)
    acc, ndcg = mo.get_acc(y_true.cpu(), lg.cpu())
    n = len(y_true)
    if not near.any():
        assert abs(res["acc1"] - acc[2, 0] / n) < 1e-12 and abs(res["acc10"] - acc[0, 0] / n) < 1e-12
        assert abs(res["ndcg5"] - ndcg[1, 0] / n) < 1e-9 and abs(res["mrr"] - mo.mrr_metric(y_true.cpu(), lg.cpu()) / n) < 1e-9
    # and within bf16 tolerance of the oracle's fp32 logits
    ref = om(ob)[0]
    assert (out["y_pred"][0].float().cpu() - ref).abs().max().item() <= 2e-2 * max(1.0, ref.abs().max().item())


def test_time_padding_row_gets_no_gradient(lib_built):
    """foursquaregraph / gowalla: time_embed_model_48 = nn.Embedding(.., padding_idx=0) (model_fqandtoyo.py:654, 796): nodes in
    slot 0 (time_normal < 1/48) read row 0 but never train it.  toyotagraph has no padding row (:915) and does train it."""
    from mobgt_b200 import synth
    for dataset_name in ("gowalla_nevda", "toyotagraph"):
        w, items, om, pm, ob, pb = _pair(dataset_name, "tiny", [(None, 6, 12, 21)])
        # force slot-0 nodes on both sides
        for it in items[:3]:
            it.time_normal[: max(1, len(it.time_normal) // 2)] = 0.0
        from mobgt_b200 import collator
        ob = mo.collate([mo.preprocess_item(it, hop_cap=20) for it in items], w, multi_hop_max_dist=20, rel_pos_max=1024)
        pb = collator.collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=1024, world=w)
        assert int((pb.slot == 0).sum()) > 0
        for m_ in (om, pm):
            m_.train()
            m_.poi_distance_model.eval()
            m_.poi_cat_model.eval()
        pm.pos_embed.p = 0.0
        om.training_loss(ob).backward()
        pm.training_step(pb).backward()
        gr, gg = om.time_embed_model_48.weight.grad, pm.time_embed_model_48.weight.grad.cpu()
        if dataset_name == "toyotagraph":
            assert gr[0].abs().max().item() > 0 and gg[0].abs().max().item() > 0
        else:
            assert gr[0].abs().max().item() == 0.0 and gg[0].abs().max().item() == 0.0
        assert (gg - gr).norm().item() <= 6e-2 * gr.norm().item()      # the smallest gradient of the model (norm 1e-4): bf16 noise


def test_k5_topk_and_rank_vs_independent_fp32(lib_built):
    """idx / cnt of the fused head against an INDEPENDENT float64 z @ W^T + bias (not the kernel's own dumped logits), on the
    rows where the comparison is decisive: the kernel accumulates exact bf16 products in fp32 (error < 2e-5 here), so top-k ids
    are compared where consecutive top-21 logits are further apart than that, ranks where no other logit is that close to the
    target's."""
    from mobgt_b200 import ops
    M, V, K, k = 256, 20011, 320, 20
    g = torch.Generator().manual_seed(2)
    z = torch.randn(M, K, generator=g).to(torch.bfloat16)
    W = (torch.randn(V, K, generator=g) * 0.05).to(torch.bfloat16)
    bias = torch.randn(V, generator=g) * 0.1
    target = torch.randint(0, V, (M,), generator=g)
    out = ops.head_topk_local(z.cuda(), W.cuda(), bias.cuda(), target.int().cuda(), k)
    logits = z.double() @ W.double().t() + bias.double()
    eps = 2e-5
    tv, ti = logits.topk(k + 1, dim=1)
    decisive = ((tv[:, :-1] - tv[:, 1:]) > eps).all(1)
    assert decisive.float().mean() > 0.8
    assert torch.equal(out["idx"].cpu().long()[decisive], ti[:, :k][decisive])
    assert (out["val"].cpu().double()[decisive] - tv[:, :k][decisive]).abs().max().item() < eps
    st = logits.gather(1, target.view(-1, 1))
    rank = (logits > st).sum(1)
    clear = ((logits - st).abs() < eps).sum(1) == 1                                 # only the target itself
    assert clear.float().mean() > 0.5
    assert torch.equal(out["cnt"].cpu().long()[clear], rank[clear])


# ------------------------------------------------------------------------------------------------------- canonical shapes
def _grad_table(ref_g, got_g):
    """per-parameter norm-wise relative error of `got_g` against `ref_g` (dicts name -> CPU fp32 gradient)"""
    gmax = max(r.abs().max().item() for r in ref_g.values())
    table = {}
    for k, r in ref_g.items():
        g = got_g.get(k)
        if g is None:
            assert r.abs().max().item() == 0.0, k
            continue
        if r.abs().max().item() < 1e-6 * gmax:            # mathematically-zero gradients (softmax ignores a per-row constant)
            assert g.abs().max().item() < 1e-3 * gmax, k
            continue
        table[k] = (g - r).norm().item() / r.norm().item()
    return table


CANONICAL = {
    # BASELINE configs[1]: toyotagraph-shaped world, 60 000 POIs, graphs at the 128-node cap + natural-law graphs in one batch
    "c2": ("toyotagraph", "c2", [(128, 10, 128, 31), (None, 6, 128, 32)]),
    # BASELINE configs[3]: gowalla_nevda-shaped world, 3 679 POIs, graphs <= 256 nodes incl. two AT 256 (T = 257: fold path)
    "c4": ("gowalla_nevda", "c4", [(256, 2, 256, 41), (None, 10, 256, 42), (130, 1, 256, 43)]),
}


@pytest.mark.parametrize("case", ["c2", "c4"])
def test_canonical_model_on_baseline_shapes(lib_built, case):
    """6 layers, ffn 1024, hidden 128, 8 heads, multi_hop_max_dist 20 (README.md:62) on BASELINE-shaped batches against the fp32
    oracle: logits and loss within 2e-2; EVERY parameter gradient within 2e-2 norm-wise — or, where twelve chained bf16 GEMM
    layers make that unreachable for ANY bf16 implementation, no worse than 2.5 x the error of the oracle itself run under
    torch.autocast(bfloat16) (the reference's `--precision 16` mixed-precision mode: Linear / matmul in 16 bit, softmax /
    LayerNorm / losses in fp32) on the same batch.  The measured table (ours | autocast) goes to gpurun_out/ and is committed
    under profiles/."""
    import copy
    dataset_name, cfg, spec = CANONICAL[case]
    w, items, om, pm, ob, pb = _pair(dataset_name, cfg, spec, n_layers=6, ffn=1024, seed=2)
    with torch.no_grad():
        ref = om(ob)
        got = pm(pb)
    for a, r in zip(got, ref):
        assert a.shape == r.shape
        assert (a.float().cpu() - r).abs().max().item() <= 2e-2 * max(1.0, r.abs().max().item())
    om16 = copy.deepcopy(om)
    gcn16 = om16.gcn_tables

    def gcn_fp32():            # torch.sparse.mm has no bf16 backward on the CPU: the GCN tables stay fp32 under autocast
        with torch.autocast("cpu", enabled=False):
            return gcn16()

    om16.gcn_tables = gcn_fp32
    for m_ in (om, om16, pm):
        m_.train()
        m_.poi_distance_model.eval()
        m_.poi_cat_model.eval()
    pm.pos_embed.p = 0.0
    lref = om.training_loss(ob)
    lref.backward()
    with torch.autocast("cpu", dtype=torch.bfloat16):
        l16 = om16.training_loss(ob)
    l16.backward()
    lgot = pm.training_step(pb)
    lgot.backward()
    assert abs(lgot.item() - lref.item()) <= 2e-2 * abs(lref.item()), (lgot.item(), lref.item())
    ref_g = {k: p.grad for k, p in om.named_parameters() if p.grad is not None}
    ours = _grad_table(ref_g, {k: p.grad.float().cpu() for k, p in pm.named_parameters() if p.grad is not None})
    auto = _grad_table(ref_g, {k: p.grad.float() for k, p in om16.named_parameters() if p.grad is not None})
    assert len(ours) > 100
    out_dir = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out_dir):
        rows = sorted(ours, key=lambda k: -ours[k])
        json.dump({"case": case, "loss": [lgot.item(), lref.item(), l16.item()],
                   "columns": ["ours vs fp32 oracle", "oracle under torch.autocast(bf16) vs fp32 oracle"],
                   "rows": {k: [round(ours[k], 5), round(auto.get(k, float("nan")), 5)] for k in rows}},
                  open(os.path.join(out_dir, f"grad_errors_{case}.json"), "w"), indent=0)
    bad = {k: (e, auto.get(k)) for k, e in ours.items() if e > max(2e-2, 2.5 * auto.get(k, 0.0))}
    assert not bad, bad


def test_bucketed_batch_matches_unpadded(lib_built):
    """A batch padded to size buckets (collator.pack_host(bucket=True): what the training loaders feed the CUDA graphs) gives
    the loss and the gradients of the unpadded batch: padding tokens belong to no graph and carry exactly zero gradient."""
    from mobgt_b200 import collator, model, synth
    w = synth.make_world("c1", seed=1, dataset_name="gowalla_nevda")
    items = synth.make_items(w, 9, 60, seed=8)
    hp = dict(n_layers=2, num_heads=8, hidden_dim=128, dropout_rate=0.0, intput_dropout_rate=0.0, weight_decay=0.01, ffn_dim=256,
              warmup_updates=10, tot_updates=100, peak_lr=2e-4, end_lr=1e-9, edge_type="multi_hop", multi_hop_max_dist=20,
              attention_dropout_rate=0.0)
    torch.manual_seed(4)
    m = model.Graphormer(dataset_name="gowalla_nevda", world=w, **hp).cuda().train()
    m.pos_embed.p = 0.0
    m.poi_distance_model.eval()
    m.poi_cat_model.eval()
    res = []
    for bucket in (False, True):
        b = collator.collate_packed(items, w, None, 512, 20, 1024, bucket=bucket)
        assert b.padded == bucket
        m.zero_grad(set_to_none=True)
        loss = m.training_step(b)
        loss.backward()
        res.append((loss.item(), {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}))
    (l0, g0), (l1, g1) = res
    assert abs(l0 - l1) <= 1e-5 * abs(l0)
    assert g0.keys() == g1.keys()
    for k in g0:
        assert torch.isfinite(g1[k]).all(), k
        scale = g0[k].abs().max().item()
        assert (g0[k] - g1[k]).abs().max().item() <= 2e-3 * scale + 1e-8, k      # other GEMM row counts -> other split-K orders


@pytest.mark.parametrize("dataset_name", ["toyotagraph", "gowalla_nevda"])
def test_gradients_written_in_place_match_autograd(lib_built, dataset_name):
    """The trainer's gradient path — every parameter gradient is a view of the flat buffer of optim.FlatAdamW; after the buffer is
    zeroed the Linear backwards WRITE into it (fp32 output of the weight-gradient GEMM, column sums and LayerNorm gradients as
    kernel outputs: ops._claim) — gives the gradients plain autograd accumulates for the same model and batch.  A second backward
    without zeroing in between ADDS (gradient accumulation keeps working)."""
    from mobgt_b200 import collator, model, ops, synth
    w = synth.make_world("c1", seed=1, dataset_name=dataset_name)
    items = synth.make_items(w, 7, 40, seed=11)
    hp = dict(n_layers=2, num_heads=8, hidden_dim=128, dropout_rate=0.0, intput_dropout_rate=0.0, weight_decay=0.01, ffn_dim=256,
              warmup_updates=10, tot_updates=100, peak_lr=2e-4, end_lr=1e-9, edge_type="multi_hop", multi_hop_max_dist=20,
              attention_dropout_rate=0.0)
    torch.manual_seed(5)
    m = model.Graphormer(dataset_name=dataset_name, world=w, **hp).cuda().train()
    m.pos_embed.p = 0.0
    m.poi_distance_model.eval()
    m.poi_cat_model.eval()
    b = collator.collate_packed(items, w, None, 512, 20, 1024)
    m.zero_grad(set_to_none=True)
    m.training_step(b).backward()                                 # plain autograd: gradients returned, bf16 dW cast to fp32
    ref = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
    (opt,), _ = m.configure_optimizers()                          # FlatAdamW: p.grad become views of opt.flat_grad
    a = m.layers[0].self_attention
    assert a.linear_k.weight.grad.data_ptr() == a.linear_q.weight.grad.data_ptr() + a.linear_q.weight.numel() * 4   # q | k | v back to back
    opt.zero_grad()
    m.training_step(b).backward()
    got = {k: p.grad.clone() for k, p in m.named_parameters()}
    assert ops._last_written.get(id(a.linear_q.weight)) == ops._zero_epoch      # the in-place path was taken
    for k, r in ref.items():
        scale = r.abs().max().item()
        assert (got[k] - r).abs().max().item() <= 6e-3 * scale + 1e-8, k         # bf16 rounding of dW on the autograd path only
    m.training_step(b).backward()                                 # no zeroing: accumulate
    for k, r in ref.items():
        scale = r.abs().max().item()
        assert (m.get_parameter(k).grad - 2 * r).abs().max().item() <= 1.5e-2 * scale + 1e-8, k


# ------------------------------------------------------------------------------------------------------- entry point
def test_entry_cli_main_reference_flags(lib_built, tmp_path, capsys):
    """`python entry.py` with the flags of the reference's README.md:62 (synthetic world instead of ../dataset): three training
    steps through the Trainer (flat gradients, PackedLoader, CUDA-graph replay of the repeated shape), a checkpoint, then
    --test from that checkpoint prints the reference's three metric lines.  Also the reference's DEFAULT --multi_hop_max_dist
    (5) runs."""
    from mobgt_b200 import entry
    common = ["--dataset_name", "toyotagraph", "--gpus", "1", "--accelerator", "ddp", "--precision", "16", "--batch_size", "16",
              "--hidden_dim", "128", "--num_heads", "8", "--n_layers", "6", "--ffn_dim", "1024", "--dropout_rate", "0.1",
              "--intput_dropout_rate", "0.1", "--attention_dropout_rate", "0.1", "--weight_decay", "0.01", "--peak_lr", "2e-4",
              "--end_lr", "1e-9", "--edge_type", "multi_hop", "--warmup_updates", "40000", "--tot_updates", "400000", "--seed", "1",
              "--max_epochs", "1", "--check_val_every_n_epoch", "1", "--synthetic", "tiny", "--train_graphs", "64", "--test_graphs",
              "40", "--n_fixed", "9"]
    root = ["--default_root_dir", str(tmp_path)]
    r = entry.cli_main(common + root + ["--multi_hop_max_dist", "20", "--limit_train_steps", "3"])
    assert r["steps"] == 3 and np.isfinite(r["loss"])
    assert os.path.exists(os.path.join(str(tmp_path), "lightning_logs", "checkpoints", "last.ckpt"))
    out = capsys.readouterr().out
    assert "CUDA-graph replays" in out
    m1 = r["metrics"]
    r2 = entry.cli_main(common + root + ["--multi_hop_max_dist", "20", "--test",
                                  "--checkpoint_path", os.path.join(str(tmp_path), "lightning_logs", "checkpoints", "last.ckpt")])
    out = capsys.readouterr().out
    assert "ACC @1:" in out and "NDCG @1:" in out and "MRR:" in out
    # same weights, same test set; a fresh process may pick other cuBLAS algorithms (last-bit differences -> a near-tie may flip)
    assert r2["metrics"]["n"] == 40 and abs(r2["metrics"]["mrr"] - m1["mrr"]) < 1e-3 * max(m1["mrr"], 1e-3)
    # the reference's default multi_hop_max_dist
    r3 = entry.cli_main(common + ["--default_root_dir", str(tmp_path / "d5"), "--limit_train_steps", "2"])
    assert r3["steps"] == 2 and np.isfinite(r3["loss"])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_entry_two_ranks_report_the_one_rank_metrics(lib_built, tmp_path):
    """`entry --test` under torch.distributed.run with 2 ranks prints the metrics of the WHOLE test set (every rank evaluates its
    share, the metric sums are all-reduced) — the same numbers as the 1-rank run of the same checkpoint; and a 2-rank training
    run of an epoch whose graph count does not split evenly finishes (equal batch counts per rank: no dead-locked all-reduce)."""
    import re
    import subprocess
    import sys
    common = ["--dataset_name", "toyotagraph", "--accelerator", "ddp", "--batch_size", "16", "--hidden_dim", "128", "--num_heads", "8",
              "--n_layers", "2", "--ffn_dim", "256", "--edge_type", "multi_hop", "--multi_hop_max_dist", "20", "--seed", "1",
              "--max_epochs", "1", "--synthetic", "tiny", "--train_graphs", "70", "--test_graphs", "41", "--default_root_dir",
              str(tmp_path)]
    env = dict(os.environ, PYTHONPATH=ROOT)
    run1 = lambda extra: subprocess.run([sys.executable, "-m", "mobgt_b200.entry"] + common + extra, capture_output=True, text=True,
                                        env=env, cwd=ROOT, timeout=600)
    run2 = lambda extra: subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                                         "--master-addr", "127.0.0.1", "--master-port", "29577", "-m", "mobgt_b200.entry"] + common + extra,
                                        capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    tr = run2([])                                                   # 70 graphs, 2 ranks, batch 16: 35 per rank -> 3 batches each
    assert tr.returncode == 0, tr.stderr[-2000:]
    assert "trained 3 steps" in tr.stdout
    ck = os.path.join(str(tmp_path), "lightning_logs", "checkpoints", "last.ckpt")
    a, b = run1(["--test", "--checkpoint_path", ck]), run2(["--test", "--checkpoint_path", ck])
    assert a.returncode == 0 and b.returncode == 0, (a.stderr[-1500:], b.stderr[-1500:])
    nums = lambda out: [float(x) for line in out.splitlines() if line.startswith(("ACC", "NDCG", "MRR")) for x in re.findall(r"[-+]?\d*\.\d+", line)]
    na, nb = nums(a.stdout), nums(b.stdout)
    assert len(na) == 7 and len(nb) == 7, (a.stdout, b.stdout)
    assert all(abs(x - y) <= 2e-3 for x, y in zip(na, nb)), (na, nb)
    assert "'n': 41" in a.stdout and "'n': 41" in b.stdout            # all 41 test graphs counted once
