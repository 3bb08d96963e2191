"""Head dim 16: `Graphormer(num_heads=8, hidden_dim=64)` (encoder width 64 + 32 + 32 = 128, 16 per head).

CPU: which (num_heads, hidden_dim) pairs the constructor accepts, and the head_dim check of the _hd attention entry points.
GPU: the d = 16 attention kernels (tensor-core forward / both backwards, the small-graph SIMT kernels, the fp32 kernels) against
float64 / fp32 torch references, and the whole model at hidden_dim 64 against the oracle (oracle/model_oracle.py) in both
precisions, the fused K5 head at K = 192, and `entry` training with CUDA graphs.  Tolerances are those of the d = 24 tests
(tests/test_k2_k3_k4.py, tests/test_round2_gpu.py, tests/test_fp32_mode.py), written where they are applied."""
import copy
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import model_oracle as mo  # noqa: E402

D16 = 16
H = 8


def _hp(hidden_dim=64, num_heads=8, n_layers=2, ffn=256, dk=20, **kw):
    hp = dict(n_layers=n_layers, num_heads=num_heads, hidden_dim=hidden_dim, dropout_rate=0.0, intput_dropout_rate=0.0,
              weight_decay=0.01, ffn_dim=ffn, warmup_updates=10, tot_updates=100, peak_lr=2e-4, end_lr=1e-9, edge_type="multi_hop",
              multi_hop_max_dist=dk, attention_dropout_rate=0.0)
    hp.update(kw)
    return hp


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("num_heads,hidden_dim", [(8, 64), (8, 128)])
def test_constructor_accepts_built_shapes(num_heads, hidden_dim):
    from mobgt_b200 import model, synth
    w = synth.make_world("tiny", seed=1)
    m = model.Graphormer(dataset_name="toyotagraph", world=w, **_hp(hidden_dim, num_heads))
    a = m.layers[0].self_attention
    assert a.att_size == (hidden_dim + 64) // num_heads and a.scale == a.att_size ** -0.5
    assert m.final_ln.normalized_shape == (2 * hidden_dim + 64,)


@pytest.mark.parametrize("num_heads,hidden_dim", [(8, 96), (4, 128), (32, 512)])
def test_constructor_rejects_other_shapes(num_heads, hidden_dim):
    """(8, 96): head dim 20; (4, 128): head dim 48 on 4 heads; (32, 512): the CLI defaults of add_model_specific_args."""
    from mobgt_b200 import model, synth
    w = synth.make_world("tiny", seed=1)
    with pytest.raises(NotImplementedError) as e:
        model.Graphormer(dataset_name="toyotagraph", world=w, **_hp(hidden_dim, num_heads))
    msg = str(e.value)
    assert "(8, 64)" in msg and "(8, 128)" in msg and "8 heads" in msg and "16 and 24" in msg


def test_hd_entry_points_reject_unbuilt_head_dims(lib_built):
    """head_dim is checked before anything else: an unbuilt value returns MOBGT_ERR_UNSUPPORTED and names the built ones."""
    from mobgt_b200 import _C
    L = _C.lib()
    for hd in (0, 8, 20, 32, 48):
        for name in ("mobgt_attn_fwd_hd", "mobgt_attn_bwd_hd", "mobgt_attn_f32_fwd_hd", "mobgt_attn_f32_bwd_hd"):
            argt = _C.SIGNATURES[name]
            args = [None if t is ctypes.c_void_p else 0 for t in argt]
            args[-2] = hd                                      # (..., head_dim, stream)
            assert getattr(L, name)(*args) == -3, (name, hd)  # MOBGT_ERR_UNSUPPORTED
            assert "16 and 24" in _C.last_error(), (name, _C.last_error())


# ---------------------------------------------------------------------------------------------------------------- GPU kernels
def _batch(sizes, seed=60):
    """one graph of n nodes (n + 1 tokens) per entry of sizes"""
    from mobgt_b200 import collator, synth
    w = synth.make_world("c1", seed=1)
    items = []
    for k, n in enumerate(sizes):
        items += synth.make_items(w, 1, 512, seed=seed + k, n_fixed=n, start=k)
    return collator.collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=1024, world=w)


def _bias(b, dtype=torch.bfloat16, seed=9):
    from mobgt_b200 import ops
    from test_k2_k3_k4 import tables
    R, Pp, E, W, t = tables(seed=seed)
    cu = [x.cuda().contiguous() for x in (R, Pp, E, W.view(-1), t.view(-1))]
    return ops.bias_fwd_raw(b, *cu, out_dtype=dtype)


# every path: <= 16 tokens (SIMT), 17..128 (one tile), 129 (single-token tail), 130..257 and 513 (general backward, several
# tiles), plus enough 17..61-token graphs that the 8 heads give more than 296 (graph, head) items: the persistent forward loops
MIXED = [3, 9, 15, 16, 60, 127, 128, 129, 200, 256, 512] + [16 + (7 * k) % 45 for k in range(30)]
SMALL_BOX = [1, 7, 15, 16, 40, 100, 127, 128, 128, 64]      # every graph <= 129 tokens: mode 2 takes the single-box backward


def _ref64(qkv, bias, tok_off, drop=None):
    """float64 attention (out, lse) on the bf16-rounded inputs, differentiable in qkv and bias"""
    from helpers import attn_drop_keep
    D = H * D16
    outs, lses = [], []
    for g in range(len(tok_off) - 1):
        a, e = int(tok_off[g]), int(tok_off[g + 1])
        T = e - a
        q, k, v = (qkv[a:e, i * D:(i + 1) * D].view(T, H, D16).transpose(0, 1) for i in range(3))
        s = (q * D16 ** -0.5) @ k.transpose(1, 2) + bias[g, :, :T, :T]
        lses.append(torch.logsumexp(s, -1).t())
        pr = torch.softmax(s, -1)
        if drop is not None:
            masks = [attn_drop_keep(g * H + h, T, drop[0], drop[1]) for h in range(H)]
            keep = torch.from_numpy(np.stack([m[0] for m in masks]))
            pr = pr * keep.to(pr.dtype) * masks[0][1]
        outs.append((pr @ v).transpose(0, 1).reshape(T, D))
    return torch.cat(outs), torch.cat(lses)


@pytest.mark.gpu
def test_d16_batch_covers_every_path(lib_built):
    b = _batch(MIXED)
    t = np.diff(b.tok_off.cpu().numpy())
    assert t.min() <= 16 and ((t > 16) & (t <= 128)).any() and (t == 129).any() and ((t >= 130) & (t <= 257)).any()
    assert (t == 513).any() and int((t > 16).sum()) * H > 296


@pytest.mark.gpu
def test_d16_forward_matches_float64(lib_built):
    from mobgt_b200 import ops
    b = _batch(MIXED)
    bias = _bias(b)
    ntok = int(b.tok_pos.numel())
    gen = torch.Generator().manual_seed(11)
    qkv = (torch.randn(ntok, 3 * H * D16, generator=gen) * 1.5).to(torch.bfloat16)
    tok_off = b.tok_off.cpu().numpy()
    for p, seed in ((0.0, 0), (0.1, 0x9E3779B97F4A7C15)):
        out, lse = ops.attn_fwd_raw(qkv.cuda(), bias, b, drop_p=p, seed=seed)
        torch.cuda.synchronize()
        assert out.shape == (ntok, H * D16)
        ref, ref_lse = _ref64(qkv.double(), bias.double().cpu(), tok_off, drop=(p, seed) if p > 0 else None)
        err = (out.double().cpu() - ref).abs().max().item()
        assert err <= 2e-2 * max(1.0, ref.abs().max().item()), (p, err)
        assert (lse.double().cpu() - ref_lse).abs().max().item() <= 2e-2, p


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.1])
def test_d16_backward_all_modes_match_float64(lib_built, p):
    """dq / dk / dv and dS in modes 0 (fp32 overwrite), 1 (fp32 accumulate) and 2 (bf16 plane) against float64 autograd with the
    same dropout mask; mode 1 adds exactly dS, mode 2 is mode 0's dS rounded once to bf16 and the same dqkv."""
    from mobgt_b200 import ops
    b = _batch(MIXED, seed=80)
    bias = _bias(b, seed=4)
    ntok = int(b.tok_pos.numel())
    gen = torch.Generator().manual_seed(21)
    qkv = (torch.randn(ntok, 3 * H * D16, generator=gen) * 1.2).to(torch.bfloat16)
    dout = torch.randn(ntok, H * D16, generator=gen).to(torch.bfloat16)
    seed = 0x0123456789ABCDEF if p > 0 else 0
    out, lse = ops.attn_fwd_raw(qkv.cuda(), bias, b, drop_p=p, seed=seed)
    db0 = torch.full(bias.shape, float("nan"), dtype=torch.float32, device="cuda")
    dq0 = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, db0, 0, drop_p=p, seed=seed)
    db1 = torch.full(bias.shape, 3.0, dtype=torch.float32, device="cuda")
    dq1 = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, db1, 1, drop_p=p, seed=seed)
    db2 = torch.full(bias.shape, float("nan"), dtype=torch.bfloat16, device="cuda")
    dq2 = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, db2, 2, drop_p=p, seed=seed)
    torch.cuda.synchronize()
    tok_off = b.tok_off.cpu().numpy()
    q64 = qkv.double().requires_grad_(True)
    b64 = bias.double().cpu().requires_grad_(True)
    ref, _ = _ref64(q64, b64, tok_off, drop=(p, seed) if p > 0 else None)
    (ref * dout.double()).sum().backward()
    gq = q64.grad
    for name, dq in (("mode0", dq0), ("mode1", dq1), ("mode2", dq2)):
        err = (dq.double().cpu() - gq).abs().max().item()
        assert err <= 2e-2 * max(1.0, gq.abs().max().item()), (name, err)
    assert torch.equal(dq0, dq1) and torch.equal(dq0, dq2)
    for g in range(len(tok_off) - 1):
        Tg = int(tok_off[g + 1] - tok_off[g])
        gb = b64.grad[g, :, :Tg, :Tg]
        got = db0[g, :, :Tg, :Tg].cpu()
        assert torch.isfinite(got).all(), g
        assert (got.double() - gb).abs().max().item() <= 2e-2 * max(1.0, gb.abs().max().item()), g
        assert torch.allclose(db1[g, :, :Tg, :Tg].cpu(), got + 3.0, rtol=1e-6, atol=1e-6), g
        assert torch.equal(db2[g, :, :Tg, :Tg].float().cpu(), got.to(torch.bfloat16).float()), g


@pytest.mark.gpu
def test_d16_single_box_and_general_backward_agree(lib_built):
    """All graphs <= 129 tokens, mode 2: k3_attn_bwd1_kernel; mode 0: the general kernel.  Same tolerance as the d = 24 test
    (test_round2_gpu.py::test_attention_bwd_single_box_variant): 1e-2 of the gradient's magnitude."""
    from mobgt_b200 import ops
    b = _batch(SMALL_BOX, seed=70)
    assert b.N <= 128
    bias = _bias(b, seed=4)
    ntok = int(b.tok_pos.numel())
    gen = torch.Generator().manual_seed(13)
    qkv = (torch.randn(ntok, 3 * H * D16, generator=gen) * 1.2).to(torch.bfloat16)
    dout = torch.randn(ntok, H * D16, generator=gen).to(torch.bfloat16)
    tok_off = b.tok_off.cpu().numpy()
    for p, seed in ((0.0, 0), (0.1, 0x0123456789ABCDEF)):
        out, lse = ops.attn_fwd_raw(qkv.cuda(), bias, b, drop_p=p, seed=seed)
        plane = torch.full(bias.shape, float("nan"), dtype=torch.bfloat16, device="cuda")
        dq2 = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, plane, 2, drop_p=p, seed=seed)
        db32 = torch.full(bias.shape, float("nan"), dtype=torch.float32, device="cuda")
        dq0 = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, db32, 0, drop_p=p, seed=seed)
        torch.cuda.synchronize()
        q64 = qkv.double().requires_grad_(True)
        b64 = bias.double().cpu().requires_grad_(True)
        ref, _ = _ref64(q64, b64, tok_off, drop=(p, seed) if p > 0 else None)
        (ref * dout.double()).sum().backward()
        gmag = max(1.0, q64.grad.abs().max().item())
        assert (dq2.double().cpu() - q64.grad).abs().max().item() <= 2e-2 * gmag, p
        assert (dq2.float() - dq0.float()).abs().max().item() <= 1e-2 * gmag, p
        for g in range(len(tok_off) - 1):
            Tg = int(tok_off[g + 1] - tok_off[g])
            gb = b64.grad[g, :, :Tg, :Tg]
            got = plane[g, :, :Tg, :Tg].float().cpu()
            assert torch.isfinite(got).all(), (p, g)
            assert (got.double() - gb).abs().max().item() <= 2e-2 * max(1.0, gb.abs().max().item()), (p, g)
            assert (got - db32[g, :, :Tg, :Tg].cpu()).abs().max().item() <= 1e-2 * max(1.0, gb.abs().max().item()), (p, g)


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [MIXED, SMALL_BOX])
def test_d16_bitwise_reproducible(lib_built, sizes):
    from mobgt_b200 import ops
    b = _batch(sizes, seed=90)
    bias = _bias(b, seed=2)
    ntok = int(b.tok_pos.numel())
    gen = torch.Generator().manual_seed(5)
    qkv = (torch.randn(ntok, 3 * H * D16, generator=gen) * 1.2).to(torch.bfloat16).cuda()
    dout = torch.randn(ntok, H * D16, generator=gen).to(torch.bfloat16).cuda()
    runs = []
    for _ in range(3):
        out, lse = ops.attn_fwd_raw(qkv, bias, b, drop_p=0.1, seed=77)
        plane = torch.empty(bias.shape, dtype=torch.bfloat16, device="cuda")
        dq = ops.attn_bwd_raw(qkv, bias, out, dout, lse, b, plane, 2, drop_p=0.1, seed=77)
        db = torch.zeros(bias.shape, dtype=torch.float32, device="cuda")
        dq0 = ops.attn_bwd_raw(qkv, bias, out, dout, lse, b, db, 0, drop_p=0.1, seed=77)
        live = torch.zeros(bias.shape, dtype=torch.bool, device="cuda")
        for g, (a, e) in enumerate(zip(b.tok_off[:-1].tolist(), b.tok_off[1:].tolist())):
            live[g, :, :e - a, :e - a] = True
        runs.append((out, lse, dq, plane[live], dq0, db))
    for r in runs[1:]:
        for x, y in zip(r, runs[0]):
            assert torch.equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [(1, 3, 7, 15, 16, 40, 127, 128, 129, 200, 256, 300)])
def test_d16_f32_kernels_match_torch(lib_built, sizes):
    """mobgt_attn_f32_fwd_hd / _bwd_hd at d = 16, T = 2 .. 301: out, dq / dk / dv and dS within 1e-5 of torch fp32 autograd, with
    and without dropout (test_fp32_mode.py's tolerance for d = 24); bitwise reproducible."""
    from mobgt_b200 import ops
    from test_k2_k3_k4 import torch_attention_diff
    TOL = 1e-5
    b = _batch(sizes, seed=170)
    bias = _bias(b, dtype=torch.float32, seed=5)
    ntok = int(b.tok_pos.numel())
    gen = torch.Generator().manual_seed(17)
    qkv = torch.randn(ntok, 3 * H * D16, generator=gen) * 1.2
    dout = torch.randn(ntok, H * D16, generator=gen)
    tok_off = b.tok_off.cpu().numpy()
    for p, seed in ((0.0, 0), (0.1, 0x0123456789ABCDEF)):
        out, lse = ops.attn_f32_fwd_raw(qkv.cuda(), bias, b, drop_p=p, seed=seed)
        db = torch.full(bias.shape, 7.0, dtype=torch.float32, device="cuda")
        dqkv = ops.attn_f32_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, db, 0, drop_p=p, seed=seed)
        torch.cuda.synchronize()
        q32 = qkv.clone().requires_grad_(True)
        b32 = bias.cpu().clone().requires_grad_(True)
        ref, _ = torch_attention_diff(q32, b32, tok_off, H=H, d=D16, drop=(p, seed) if p > 0 else None)
        (ref * dout).sum().backward()
        assert (out.cpu() - ref.detach()).abs().max().item() <= TOL * max(1.0, ref.abs().max().item()), p
        gq = q32.grad
        assert (dqkv.cpu() - gq).abs().max().item() <= TOL * max(1.0, gq.abs().max().item()), p
        for g in range(len(tok_off) - 1):
            Tg = int(tok_off[g + 1] - tok_off[g])
            gb = b32.grad[g, :, :Tg, :Tg]
            assert (db[g, :, :Tg, :Tg].cpu() - gb).abs().max().item() <= TOL * max(1.0, gb.abs().max().item()), (p, g)
            assert (db[g, :, Tg:, :] == 7.0).all() and (db[g, :, :Tg, Tg:] == 7.0).all(), (p, g)
        out2, lse2 = ops.attn_f32_fwd_raw(qkv.cuda(), bias, b, drop_p=p, seed=seed)
        db2 = torch.full(bias.shape, 7.0, dtype=torch.float32, device="cuda")
        dq2 = ops.attn_f32_bwd_raw(qkv.cuda(), bias, out2, dout.cuda(), lse2, b, db2, 0, drop_p=p, seed=seed)
        assert torch.equal(out2, out) and torch.equal(lse2, lse) and torch.equal(dq2, dqkv) and torch.equal(db2, db)


# ---------------------------------------------------------------------------------------------------------------- GPU model
# two layers; graphs from 2 to 300 nodes (every attention path) next to natural-law graphs
MODEL_CASES = {
    "toyota": ("toyotagraph", [(2, 1, 512, 51), (None, 6, 40, 52), (128, 1, 512, 53), (300, 1, 512, 54)]),
    "gowalla": ("gowalla_nevda", [(2, 1, 512, 61), (None, 6, 40, 62), (129, 1, 512, 63), (300, 1, 512, 64)]),
}


def _pair64(dataset_name, spec, seed=3, precision=16, hidden_dim=64):
    """oracle + product model at hidden_dim 64 (or the canonical 128) with the same weights, and the two batches of the same
    items"""
    from mobgt_b200 import collator, model, synth
    w = synth.make_world("c1", seed=seed, dataset_name=dataset_name)
    items = []
    for n_fixed, cnt, cap, sd in spec:
        items += synth.make_items(w, cnt, cap, seed=sd, n_fixed=n_fixed, start=len(items))
    torch.manual_seed(seed)
    om = mo.Graphormer(w, n_layers=2, num_heads=8, hidden_dim=hidden_dim, ffn_dim=256, dataset_name=dataset_name).eval()
    with torch.no_grad():
        for emb in (om.edge_encoder, om.rel_pos_encoder, om.poi_pos_encoder):
            emb.weight.mul_(0.3)
            emb.weight[0].zero_()
        om.edge_dis_encoder.weight.mul_(0.3)
    pm = model.Graphormer(dataset_name=dataset_name, world=w, precision=precision, **_hp(hidden_dim)).cuda().eval()
    missing, _ = pm.load_state_dict(om.state_dict(), strict=False)
    assert not missing, missing
    ob = mo.collate([mo.preprocess_item(it, hop_cap=20) for it in items], w, multi_hop_max_dist=20, rel_pos_max=1024)
    pb = collator.collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=1024, world=w)
    assert pb.N == 300 and min(pb.n_host) <= 15
    return om, pm, ob, pb


def _train_mode(*ms):
    for m_ in ms:
        m_.train()
        m_.poi_distance_model.eval()      # GCN dropout masks are torch's own: off, like every other dropout here
        m_.poi_cat_model.eval()


def _fp32_errors(case, hidden_dim):
    """precision=32 model against the oracle on the items of MODEL_CASES[case]: checks logits and loss within 1e-5 and returns
    {parameter: (error vs the fp32 oracle, error vs the oracle run in float64)}, norm-wise"""
    from test_fp32_mode import _oracle_float64
    TOL = 1e-5
    om, pm, ob, pb = _pair64(*MODEL_CASES[case], precision=32, hidden_dim=hidden_dim)
    with torch.no_grad():
        ref = om(ob)
        got = pm(pb)
    for a, r in zip(got, ref):
        assert a.dtype == torch.float32 and a.shape == r.shape
        assert (a.cpu() - r).abs().max().item() <= TOL * max(1.0, r.abs().max().item())
    _train_mode(om, pm)
    pm.pos_embed.p = 0.0
    lref = om.training_loss(ob)
    lref.backward()
    lgot = pm.training_step(pb)
    lgot.backward()
    assert abs(lgot.item() - lref.item()) <= TOL * abs(lref.item()), (lgot.item(), lref.item())
    ref_g = {k: p.grad for k, p in om.named_parameters() if p.grad is not None}
    got_g = {k: p.grad.float().cpu() for k, p in pm.named_parameters() if p.grad is not None}
    _, ref64_g = _oracle_float64(om, ob)
    gmax = max(r.abs().max().item() for r in ref_g.values())
    table = {}
    for k, r in ref_g.items():
        g = got_g.get(k)
        if g is None:
            assert r.abs().max().item() == 0.0, k
            continue
        if r.abs().max().item() < 1e-6 * gmax:        # mathematically-zero gradients (softmax ignores a per-row constant)
            assert g.abs().max().item() < 1e-4 * gmax, k
            continue
        r64 = ref64_g[k]
        table[k] = ((g - r).norm().item() / r.norm().item(), (g.double() - r64).norm().item() / r64.norm().item())
    return table


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(MODEL_CASES))
def test_hidden64_fp32_mode_matches_oracle(lib_built, case):
    """precision=32: logits and loss within 1e-5, every parameter gradient within 1e-5 norm-wise of the fp32 oracle, or of the
    oracle run in float64 where the fp32 oracle's own rounding is a sizeable part of 1e-5 (test_fp32_mode.py's gate).

    A gradient that misses both is compared with the canonical model (hidden_dim 128, head dim 24) on the same items: the
    head-dim-16 path must then be no worse than 2.5x the head-dim-24 path's own error against float64.  This is for the two
    edge tables on a batch with a 300-node graph: their gradients are sums over every (cell, hop) of the attention-bias
    gradient, which nearly cancel (each row of dS sums to zero), and the bias-table backward (K2, unchanged here) reduces
    them in fp32 through its rel_pos histogram, where the fp32 oracle sums cell by cell.  Measured on the B200 (gowalla case,
    norm-wise error against float64): edge_encoder 3.2e-4 at head dim 16 and 9.6e-4 at head dim 24, edge_dis_encoder 1.8e-4
    and 5.2e-4; without the 300-node graph, 1.2e-5 and 7.6e-6 at head dim 16.  Every other gradient is within 1e-5."""
    from mobgt_b200 import model
    TOL = 1e-5
    try:
        table = _fp32_errors(case, 64)
        assert len(table) > 40
        miss = {k: e for k, e in table.items() if min(e) > TOL}
        if miss:
            canon = _fp32_errors(case, 128)
            worse = {k: (e, canon.get(k)) for k, e in miss.items() if k not in canon or e[1] > 2.5 * max(canon[k][1], TOL)}
            assert not worse, worse
    finally:
        model.ops.enable_tf32(True)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(MODEL_CASES))
def test_hidden64_bf16_mode_matches_oracle(lib_built, case):
    """precision=16: logits and loss within 2e-2; every parameter gradient within 2e-2 norm-wise, or no worse than 2.5x the
    error of the oracle under torch.autocast(bfloat16) (the gate of test_round2_gpu.py::test_canonical_model_on_baseline_shapes)."""
    from test_round2_gpu import _grad_table
    om, pm, ob, pb = _pair64(*MODEL_CASES[case])
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
    _train_mode(om, om16, pm)
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
    assert len(ours) > 40
    bad = {k: (e, auto.get(k)) for k, e in ours.items() if e > max(2e-2, 2.5 * auto.get(k, 0.0))}
    assert not bad, bad


@pytest.mark.gpu
def test_hidden64_head_topk_k192(lib_built):
    """Graphormer.head_topk at hidden_dim 64: the fused K5 head runs at K = 2 * 64 + 64 = 192.  Top-k ids and the target ranks
    against an independent fp32 product of the same bf16 operands.  Both sum exact bf16 products in fp32, in different orders:
    ids are compared on the rows whose 21 largest logits are more than EPS apart, ranks within the +-EPS tie window."""
    from mobgt_b200 import model, synth
    w = synth.make_world("c2", seed=1, dataset_name="gowalla_nevda")
    pm = model.Graphormer(dataset_name="gowalla_nevda", world=w, **_hp(64)).cuda().eval()
    assert pm.out_proj.in_features == 192
    g = torch.Generator().manual_seed(3)
    M, k = 300, 20
    z = (torch.randn(M, 192, generator=g) * 3).cuda()
    EPS = 1e-4
    y = torch.randint(0, pm.out_proj.out_features, (M,), generator=g).cuda()
    r = pm.head_topk(z, y, k)
    torch.cuda.synchronize()
    W = pm.out_proj.weight.detach().to(torch.bfloat16).float()
    logits = z.to(torch.bfloat16).float() @ W.t() + pm.out_proj.bias.detach().float()
    tv, ti = logits.topk(k + 1, dim=1)
    assert (r["val"].float() - tv[:, :k]).abs().max().item() <= 2e-3 * max(1.0, tv.abs().max().item())
    sep = (tv[:, :k] - tv[:, 1:]).min(1).values > EPS                                          # rows without near-ties
    assert int(sep.sum()) > M // 2
    assert torch.equal(r["idx"].long()[sep], ti[sep, :k])
    st = logits.gather(1, y.view(-1, 1))
    lo = (logits > st + EPS).sum(1)
    hi = (logits >= st - EPS).sum(1) - 1
    rank = r["rank"].long()
    assert ((rank >= lo) & (rank <= hi)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [16, 32])
def test_hidden64_entry_trains_and_tests(lib_built, precision, tmp_path):
    """`entry --hidden_dim 64 --num_heads 8`: a few training steps (precision 16: CUDA-graph capture and replay of the bucketed
    step), a finite loss, then `--test` on the checkpoint returns the metric dict."""
    from mobgt_b200 import entry, model
    common = ["--dataset_name", "toyotagraph", "--gpus", "1", "--precision", str(precision), "--batch_size", "16",
              "--hidden_dim", "64", "--num_heads", "8", "--n_layers", "2", "--ffn_dim", "256", "--dropout_rate", "0.1",
              "--intput_dropout_rate", "0.1", "--attention_dropout_rate", "0.1", "--weight_decay", "0.01", "--peak_lr", "2e-4",
              "--end_lr", "1e-9", "--edge_type", "multi_hop", "--warmup_updates", "40000", "--tot_updates", "400000", "--seed",
              "1", "--max_epochs", "1", "--synthetic", "tiny", "--train_graphs", "96", "--test_graphs", "24",
              "--multi_hop_max_dist", "20", "--default_root_dir", str(tmp_path)]
    try:
        r = entry.cli_main(common + ["--limit_train_steps", "5"])
        assert r["steps"] == 5 and np.isfinite(r["loss"])
        if precision == 16:
            assert r["graph_steps"] >= 1, r
        ck = [os.path.join(dp, f) for dp, _, fs in os.walk(tmp_path) for f in fs if f == "last.ckpt"]
        assert len(ck) == 1
        t = entry.cli_main(common + ["--test", "--resume_from_checkpoint", ck[0]])
        m = t["metrics"]
        assert m["n"] == 24 and all(np.isfinite(m[k_]) for k_ in ("acc1", "acc5", "acc10", "acc20", "mrr"))
    finally:
        model.ops.enable_tf32(True)
