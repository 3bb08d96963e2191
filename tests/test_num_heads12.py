"""12 heads: `Graphormer(num_heads=12, hidden_dim=128)` (encoder width 128 + 32 + 32 = 192, 16 per head).

CPU: which shapes the constructor accepts, the head-count check of the K2 entry points, an H-generic float64 K2 reference pinned
to the oracle's attn_bias_build at 12 heads, and a Python copy of the 12-head backward plan checked against the library's
workspace size.
GPU: the 12-head K2 kernels (forward fp32 / bf16, backward from one fp32 plane or 1 / 6 / 7 bf16 layer planes) against that
reference on adversarial packed batches (tests/test_k2_bias_adversarial.py, whose tolerances apply), the attention kernels (K3)
at H = 12 against float64 attention, the whole model at (12, 128) against the oracle (oracle/model_oracle.py) in both
precisions, and `entry` training with CUDA graphs."""
import copy
import ctypes
import os

import numpy as np
import pytest
import torch

import model_oracle as mo
from test_k2_bias_adversarial import (GRAD_NAMES, SMALLS, _chain_item, _packed_from_oracle, adversarial_batch, expected_walk,
                                      live_mask, pair_index)

H = 12
D16 = 16
NEG_INF = float("-inf")


def _hp(num_heads=12, hidden_dim=128, n_layers=2, ffn=256, dk=20, **kw):
    hp = dict(n_layers=n_layers, num_heads=num_heads, hidden_dim=hidden_dim, dropout_rate=0.0, intput_dropout_rate=0.0,
              weight_decay=0.01, ffn_dim=ffn, warmup_updates=10, tot_updates=100, peak_lr=2e-4, end_lr=1e-9, edge_type="multi_hop",
              multi_hop_max_dist=dk, attention_dropout_rate=0.0)
    hp.update(kw)
    return hp


# ---------------------------------------------------------------------------------------------------------------- reference
def k2_reference_h(n, rel_pos, poi_pos, edge_in, dk, rel_pos_max, R, Ppos, E, W, tvd):
    """test_k2_bias_adversarial.k2_reference for any head count (H = R.shape[1]): dense bias [B, H, T, T] from packed indices,
    differentiable in the five tables."""
    n = [int(v) for v in n]
    nh = R.shape[1]
    B, T = len(n), max(n) + 1
    rp, pp, ei = (torch.as_tensor(x).long() for x in (rel_pos, poi_pos, edge_in))
    W3 = W.reshape(-1, nh, nh)
    e = torch.zeros(rp.numel(), nh, dtype=R.dtype)
    for k in range(dk):
        e = e + (E @ W3[k])[ei[:, k]]
    sp = (rp - 1).clamp(1, dk).to(R.dtype)
    val = R[rp] + Ppos[pp] + e / sp[:, None]
    val = torch.where(((rp - 1) >= rel_pos_max)[:, None], torch.full_like(val, NEG_INF), val)
    g, i, j = pair_index(n)
    out = torch.zeros(B, nh, T, T, dtype=R.dtype)
    out[g, :, i + 1, j + 1] = val
    for gi, k in enumerate(n):
        out[gi, :, 1:k + 1, 0] = tvd.reshape(nh, 1)
    return out


def _tables(bins, hops, seed, scale=0.3):
    g = torch.Generator().manual_seed(seed)
    R = torch.randn(512, H, generator=g, dtype=torch.float64) * scale
    Pp = torch.randn(bins, H, generator=g, dtype=torch.float64) * scale
    E = torch.randn(128, H, generator=g, dtype=torch.float64) * scale
    W = torch.randn(hops * H * H, generator=g, dtype=torch.float64) * scale
    t = torch.randn(H, generator=g, dtype=torch.float64) * scale
    E[0] = 0
    return R, Pp, E, W, t


def _reference_grads(pk, tabs, dB):
    leaves = [t.detach().double().clone().requires_grad_(True) for t in tabs]
    out = k2_reference_h(pk.n_host, pk.h_rel, pk.h_poi, pk.h_edge, pk.dk, pk.rel_pos_max, *leaves)
    fin = torch.isfinite(out)
    (torch.where(fin, out, torch.zeros_like(out)) * dB).sum().backward()
    return [lf.grad for lf in leaves]


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_constructor_accepts_12_heads_128():
    from mobgt_b200 import model, synth
    w = synth.make_world("tiny", seed=1)
    m = model.Graphormer(dataset_name="toyotagraph", world=w, **_hp())
    a = m.layers[0].self_attention
    assert a.num_heads == 12 and a.att_size == 16 and a.scale == 16 ** -0.5
    assert a.linear_q.out_features == 192 and m.final_ln.normalized_shape == (320,) and m.out_proj.in_features == 320
    for emb in (m.edge_encoder, m.rel_pos_encoder, m.poi_pos_encoder, m.graph_token_virtual_distance):
        assert emb.weight.shape[1] == 12
    assert m.edge_dis_encoder.weight.shape == (128 * 12 * 12, 1)


@pytest.mark.parametrize("num_heads,hidden_dim", [(12, 64), (12, 224), (16, 192), (16, 128)])
def test_constructor_rejects_other_12_and_16_head_shapes(num_heads, hidden_dim):
    """(12, 64): head dim 32 / 3; (12, 224): head dim 24 but a 512-wide LayerNorm; (16, 192): head dim 16 but a 448-wide
    LayerNorm / K5 head; (16, 128): head dim 12."""
    from mobgt_b200 import model, synth
    w = synth.make_world("tiny", seed=1)
    with pytest.raises(NotImplementedError) as e:
        model.Graphormer(dataset_name="toyotagraph", world=w, **_hp(num_heads, hidden_dim))
    msg = str(e.value)
    assert "(8, 64)" in msg and "(8, 128)" in msg and "(12, 128)" in msg and "8 heads" in msg and "12 heads" in msg
    assert "16 and 24" in msg


def test_k2_entry_points_reject_unbuilt_head_counts(lib_built):
    """num_heads is checked before anything else: 4, 16 and 32 return MOBGT_ERR_UNSUPPORTED naming 8 and 12; the workspace
    queries return < 0.  The 3-argument backward workspace query is the 8-head one."""
    from mobgt_b200 import _C
    L = _C.lib()
    for nh in (4, 16, 32):
        for name, pos in (("mobgt_bias_fwd", 10), ("mobgt_bias_bwd", 10)):
            argt = _C.SIGNATURES[name]
            args = [None if t is ctypes.c_void_p else 0 for t in argt]
            args[pos] = nh                                    # (..., hops, dk, H, rel_pos_max, ...)
            assert getattr(L, name)(*args) == -3, (name, nh)
            assert "8 and 12" in _C.last_error(), (name, _C.last_error())
        assert L.mobgt_bias_fwd_workspace_bytes(20, nh) < 0
        assert L.mobgt_bias_bwd_heads_workspace_bytes(129, 20, 64, nh) < 0
    for T, hops, bins in ((2, 4, 1), (129, 20, 64), (513, 32, 1024)):
        assert L.mobgt_bias_bwd_heads_workspace_bytes(T, hops, bins, 8) == L.mobgt_bias_bwd_workspace_bytes(T, hops, bins) > 0
        assert L.mobgt_bias_bwd_heads_workspace_bytes(T, hops, bins, 12) > 0
    assert L.mobgt_bias_fwd_workspace_bytes(20, 12) == (20 * 128 + 512) * 12 * 4


@pytest.mark.parametrize("rel_pos_max", [1024, 20, 3])
@pytest.mark.parametrize("dk", [5, 20])
def test_reference_equals_oracle_attn_bias_build_12_heads(rel_pos_max, dk):
    """k2_reference_h at 12 heads == model_oracle.Graphormer.attn_bias_build run in float64 with 12-column tables on an
    oracle-collated batch: finite cells within 1e-12 of the cell's magnitude bound, identical -inf sets."""
    from mobgt_b200 import synth
    w = synth.make_world("c1", seed=1)
    items = synth.make_items(w, 5, 40, seed=dk + rel_pos_max) + [_chain_item(w, 33, 7, 5), _chain_item(w, 4, 8, 6)]
    ob = mo.collate([mo.preprocess_item(it, hop_cap=max(20, dk)) for it in items], w, multi_hop_max_dist=dk, rel_pos_max=rel_pos_max)
    R, Pp, E, W, t = _tables(w.num_bins, 20, seed=dk)
    R[0] = 0
    Pp[0] = 0
    m = mo.Graphormer.__new__(mo.Graphormer)
    torch.nn.Module.__init__(m)
    m.num_heads, m.multi_hop_max_dist = H, dk
    m.rel_pos_encoder = torch.nn.Embedding.from_pretrained(R.clone(), freeze=False, padding_idx=0)
    m.poi_pos_encoder = torch.nn.Embedding.from_pretrained(Pp.clone(), freeze=False, padding_idx=0)
    m.edge_encoder = torch.nn.Embedding.from_pretrained(E.clone(), freeze=False, padding_idx=0)
    m.edge_dis_encoder = torch.nn.Embedding.from_pretrained(W.view(-1, 1).clone(), freeze=False)
    m.graph_token_virtual_distance = torch.nn.Embedding.from_pretrained(t.view(1, -1).clone(), freeze=False)
    ob64 = copy.copy(ob)
    ob64.attn_bias = ob.attn_bias.double()
    with torch.no_grad():
        orc = m.attn_bias_build(ob64, "fp32")
    assert orc.dtype == torch.float64
    n, rel, poi, edge = _packed_from_oracle(ob, dk)
    ref = k2_reference_h(n, rel, poi, edge, dk, rel_pos_max, R, Pp, E, W, t)
    A = k2_reference_h(n, rel, poi, edge, dk, rel_pos_max, R.abs(), Pp.abs(), E.abs(), W.abs(), t.abs())
    T = max(n) + 1
    assert orc.shape == ref.shape == (len(n), H, T, T)
    live = live_mask(n, T).expand_as(ref)
    o, r, a = orc[live], ref[live], A[live]
    assert torch.equal(torch.isneginf(o), torch.isneginf(r))
    fin = torch.isfinite(r)
    assert ((o[fin] - r[fin]).abs() <= 1e-12 * a[fin]).all()
    if rel_pos_max < 1024:
        assert torch.isneginf(r).any() and fin.any()


def k2_bwd_plan12(T, hops, num_bins):
    """Python restatement of k2_bwd_plan<12> (csrc/k2_bias.cu): (histogram rows, partial-row stride, warps per CTA).  At 12
    heads the histograms have ONE cell slot (K2Heads<12>::kSlots), the dsum strip 12 head rows."""
    rrows = min(T, 511) + 1
    nR, nP = rrows * H, num_bins * H
    stride = hops * 16 * H + nR + nP + H
    pitch = ((((T + 3) & ~3) + 27) // 32) * 32 + 4
    per_warp = (nR + H) + (nP + H) + H * pitch + 3 * pitch + H
    cta_words = (hops + 1) * 8 + 40
    return rrows, stride, min((227 * 1024 - 2048 - cta_words * 4) // (per_warp * 4), 12)


# (hops, dk, graph sizes, num_bins, rel_pos_max, extra pitch, bf16 layer planes, backward warps planned at 12 heads)
K2_CASES12 = [
    (4, 4, [1], 64, 1024, 0, 1, 12),                    # T = 2
    (4, 1, [2, 3, 1, 3], 1, 20, 0, 6, 12),              # T = 4
    (8, 8, [12, 5, 1, 9], 1024, 3, 0, 7, 4),            # T = 13
    (8, 3, [13, 2, 7], 64, 1024, 0, 6, 12),             # T = 14
    (12, 12, [14, 14, 3], 1, 1024, 0, 7, 12),           # T = 15
    (12, 5, [15, 8, 1], 1024, 20, 0, 1, 4),             # T = 16
    (16, 16, [16, 4, 11, 16], 64, 3, 0, 6, 12),         # T = 17
    (16, 1, [17, 2], 64, 1024, 24, 7, 12),              # T = 18, pitch 48 > round_up(T, 8)
    (20, 20, [18, 9, 3], 1024, 1024, 0, 1, 4),          # T = 19
    (20, 7, [35, 20, 6], 64, 20, 0, 6, 12),             # T = 36
    (8, 8, [47, 3, 3], 1, 1024, 0, 7, 12),              # T = 48
    (24, 13, [128, 64, 3], 1024, 1024, 0, 6, 3),        # T = 129
    (20, 20, [200, 1, 2], 1, 1024, 0, 7, 9),            # T = 201
    (24, 24, [299, 150, 40, 7], 64, 1024, 0, 1, 6),     # T = 300
    (28, 2, [509, 12], 64, 20, 0, 7, 3),                # T = 510: key 510 is the only one past the plan
    (32, 32, [510, 30], 1, 1024, 0, 6, 4),              # T = 511
    (28, 28, [512] + SMALLS, 1024, 1024, 0, 6, 2),      # T = 513: one 512-node graph and many small ones
    (32, 17, [512] + SMALLS, 64, 3, 0, 1, 3),           # T = 513
]


def _case_id(c):
    return f"h{c[0]}-dk{c[1]}-T{max(c[2]) + 1}-bins{c[3]}-rpm{c[4]}"


def test_case_matrix_12_heads(lib_built):
    """Every hop width with dk = hops and dk < hops, every T residue mod 8, all rel_pos_max and num_bins values; the 12-head
    plan of each case as asserted, its row layout equal to the library's workspace size.  The warp counts the cases reach
    are 2, 3, 4, 6, 9 and 12 (8 heads at the same T / bins: 1, 2, 3, 4, 6, 9, 12)."""
    from mobgt_b200 import _C
    L = _C.lib()
    assert {c[0] for c in K2_CASES12} == {4, 8, 12, 16, 20, 24, 28, 32}
    for hops in range(4, 33, 4):
        dks = {c[1] for c in K2_CASES12 if c[0] == hops}
        assert hops in dks and min(dks) < hops
    assert 1 in {c[1] for c in K2_CASES12}
    assert {(max(c[2]) + 1) % 8 for c in K2_CASES12} == set(range(8))
    assert {c[4] for c in K2_CASES12} == {1024, 20, 3} and {c[3] for c in K2_CASES12} == {1, 64, 1024}
    assert {c[6] for c in K2_CASES12} == {1, 6, 7}
    warps = set()
    for hops, dk, ns, bins, rpm, extra, layers, want in K2_CASES12:
        T = max(ns) + 1
        rrows, stride, got = k2_bwd_plan12(T, hops, bins)
        assert got == want, (hops, ns, bins, got, want)
        warps.add(got)
        # workspace = dEW + (SMs + 1) partial rows + 16 + SMs per-CTA fixed-point tables + the launch-wide fixed-point tables
        ws = int(L.mobgt_bias_bwd_heads_workspace_bytes(T, hops, bins, H))
        rest = ws - 16 - 4 * hops * 128 * H - 8 * (hops * 128 * H + 512 * H) - 4 * stride
        assert ws > 0 and rest > 0 and rest % (4 * stride + 8 * hops * 16 * H) == 0, (hops, T, bins)
    assert {2, 3, 4, 6, 9, 12} <= warps, warps
    # the warps per CTA at T = 129 and T = 513 (hops 20, bins 1024) next to the 8-head plan (test_k2_bias_adversarial)
    from test_k2_bias_adversarial import k2_bwd_plan
    assert [k2_bwd_plan12(T, 20, 1024)[2] for T in (129, 513)] == [3, 2]
    assert [k2_bwd_plan(T, 20, 1024)[2] for T in (129, 513)] == [2, 1]


# ---------------------------------------------------------------------------------------------------------------- GPU: K2
def _bwd_call(pk, dbias, dtype_code, n_layers, layer_stride, T, Tp, E, W, num_bins):
    """mobgt_bias_bwd at 12 heads through the C-ABI with an explicit plane stride"""
    from mobgt_b200 import _C
    dev = E.device
    ws_bytes = int(_C.lib().mobgt_bias_bwd_heads_workspace_bytes(T, pk.hops, num_bins, H))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    dR = torch.empty(512, H, device=dev)
    dP = torch.empty(num_bins, H, device=dev)
    dE = torch.empty(128, H, device=dev)
    dW = torch.zeros(W.numel(), device=dev)
    dt = torch.empty(H, device=dev)
    _C.call("mobgt_bias_bwd", _C.ptr(pk.n), _C.ptr(pk.sq_off), _C.ptr(pk.rel_pos16), _C.ptr(pk.poi_pos16), _C.ptr(pk.edge_in8),
            pk.B, T, Tp, pk.hops, pk.dk, H, pk.rel_pos_max, num_bins, dbias.data_ptr(), dtype_code, n_layers, layer_stride,
            _C.ptr(E), _C.ptr(W), _C.ptr(ws), ws_bytes, _C.ptr(dR), _C.ptr(dP), _C.ptr(dE), _C.ptr(dW), _C.ptr(dt), _C.stream_ptr())
    return dR, dP, dE, dW, dt


def _check_grads(got, ref, A, tag):
    for name, g, r, a in zip(GRAD_NAMES, got, ref, A):
        g = g.detach().double().cpu().reshape(r.shape)
        if name == "dE":
            assert (g[0] == 0).all(), tag
            g, r, a = g[1:], r[1:], a[1:]
        err = (g - r).abs()
        bad = err > 2e-5 * a
        assert not bad.any(), (tag, name, int(bad.sum()), float(err.max()), float((err / a.clamp_min(1e-300)).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("case", K2_CASES12, ids=_case_id)
def test_k2_12_heads_fwd_bwd_matches_float64(lib_built, case):
    """mobgt_bias_fwd (fp32, bf16) and mobgt_bias_bwd (one fp32 plane; n_layers bf16 planes, contiguous and, for 6 and 7
    planes, spaced wider than one plane) at 12 heads against k2_reference_h in float64, with the tolerances of
    test_k2_bias_adversarial.py; NaN in the dBias cells the kernel must not read changes no bit."""
    from mobgt_b200 import ops
    hops, dk, ns, bins, rpm, extra, n_layers, want_warps = case
    seed = hops * 1000 + dk * 10 + len(ns) + 7
    pk = adversarial_batch(seed, ns, hops, dk, bins, rpm)
    T = pk.N + 1
    Tp = ops.bias_pitch(T) + extra
    assert k2_bwd_plan12(T, hops, bins)[2] == want_warps
    tabs = _tables(bins, hops, seed)
    A_tabs = [x.abs() for x in tabs]
    ref = k2_reference_h(pk.n_host, pk.h_rel, pk.h_poi, pk.h_edge, dk, rpm, *tabs)
    A = k2_reference_h(pk.n_host, pk.h_rel, pk.h_poi, pk.h_edge, dk, rpm, *A_tabs)
    live = live_mask(pk.n_host, T).expand_as(ref)
    masked = torch.isneginf(ref) & live
    fin = live & ~masked
    kk = pk.h_rel
    nd = (pk.h_edge != torch.from_numpy(np.where(np.arange(hops)[None, :] < expected_walk(kk.numpy(), dk)[:, None], 4, 0))).sum(1)
    if max(ns) > 1:
        assert (kk == 511).any() and ((kk >= 2) & (kk < 511)).any()
        assert (nd == 0).any() and (nd >= 1).any()
    if max(ns) + 1 < 511 and max(ns) > 20:
        assert (kk >= T).any() and (kk < 511).any()          # keys past the backward's histogram plan
    cu = [x.float().cuda().contiguous() for x in tabs]
    for dt in (torch.float32, torch.bfloat16):
        out = ops.bias_fwd_raw(pk, *cu, out_dtype=dt, T=T, Tp=Tp)
        assert out.shape == (pk.B, H, T, Tp)
        got = out[..., :T].double().cpu()
        assert torch.isneginf(got[masked]).all(), dt
        g, r, a = got[fin], ref[fin], A[fin]
        assert torch.isfinite(g).all(), dt
        tol = 1e-5 * a if dt == torch.float32 else 2.0 ** -8 * r.abs() + 1e-5 * a
        bad = (g - r).abs() > tol
        assert not bad.any(), (dt, int(bad.sum()), float((g - r).abs().max()))
    gen = torch.Generator().manual_seed(seed + 1)
    sq = live_mask(pk.n_host, T, Tp).expand(pk.B, H, T, Tp)
    dB = torch.where(sq, torch.randn(pk.B, H, T, Tp, generator=gen), torch.zeros(()))
    used = torch.zeros(pk.B, H, T, Tp, dtype=torch.bool)
    used[..., :T] = fin
    used[:, :, 0, :] = False
    Ecu, Wcu = cu[2], cu[3]
    dB64 = dB[..., :T].double()
    got32 = ops.bias_bwd_raw(pk, dB.cuda(), Ecu, Wcu, bins)
    _check_grads(got32, _reference_grads(pk, tabs, dB64), _reference_grads(pk, A_tabs, dB64.abs()), "f32")
    dirty = torch.where(used, dB, torch.full((), float("nan")))
    again = ops.bias_bwd_raw(pk, dirty.cuda(), Ecu, Wcu, bins)
    for a_, b_, name in zip(again, got32, GRAD_NAMES):
        assert torch.equal(a_, b_), ("f32 NaN fill", name)
    planes = torch.stack([(torch.randn(pk.B, H, T, Tp, generator=gen) * (0.5 + 0.25 * l)).to(torch.bfloat16)
                          for l in range(n_layers)])
    planes = torch.where(sq.unsqueeze(0), planes, torch.zeros((), dtype=torch.bfloat16))
    got16 = ops.bias_bwd_raw(pk, planes.cuda(), Ecu, Wcu, bins)
    _check_grads(got16, _reference_grads(pk, tabs, planes.double().sum(0)[..., :T]),
                 _reference_grads(pk, A_tabs, planes.double().abs().sum(0)[..., :T]), f"bf16 x{n_layers}")
    nanbf = torch.full((), float("nan"), dtype=torch.bfloat16)
    dirty16 = torch.where(used.unsqueeze(0), planes, nanbf)
    again16 = ops.bias_bwd_raw(pk, dirty16.cuda(), Ecu, Wcu, bins)
    for a_, b_, name in zip(again16, got16, GRAD_NAMES):
        assert torch.equal(a_, b_), ("bf16 NaN fill", name)
    if n_layers in (6, 7):
        plane = pk.B * H * T * Tp
        ls = plane + 40
        flat = torch.full((n_layers * ls,), float("nan"), dtype=torch.bfloat16)
        flat.view(n_layers, ls)[:, :plane] = dirty16.reshape(n_layers, plane)
        gs = _bwd_call(pk, flat.cuda(), ops.BF16, n_layers, ls, T, Tp, Ecu, Wcu, bins)
        for a_, b_, name in zip(gs, got16, GRAD_NAMES):
            assert torch.equal(a_, b_), ("bf16 strided", name)


@pytest.mark.gpu
def test_k2_12_heads_backward_bitwise_reproducible(lib_built):
    """Rare path (deviating bytes, features >= 16, keys past the plan) at 12 heads: three repeats give identical bits, from an
    fp32 buffer and from 7 bf16 planes; the forward repeats bit for bit too."""
    from mobgt_b200 import ops
    hops, dk, bins = 24, 24, 64
    pk = adversarial_batch(98, [200, 150, 90, 60, 33, 17, 9], hops, dk, bins, 1024)
    T = pk.N + 1
    Tp = ops.bias_pitch(T)
    tabs = [x.float().cuda().contiguous() for x in _tables(bins, hops, 98)]
    f0 = ops.bias_fwd_raw(pk, *tabs, out_dtype=torch.bfloat16)
    gen = torch.Generator().manual_seed(6)
    sq = live_mask(pk.n_host, T, Tp).expand(pk.B, H, T, Tp)
    dB = torch.where(sq, torch.randn(pk.B, H, T, Tp, generator=gen), torch.zeros(())).cuda()
    planes = torch.where(sq.unsqueeze(0), torch.randn(7, pk.B, H, T, Tp, generator=gen), torch.zeros(())).to(torch.bfloat16).cuda()
    for src in (dB, planes):
        first = ops.bias_bwd_raw(pk, src, tabs[2], tabs[3], bins)
        for _ in range(3):
            again = ops.bias_bwd_raw(pk, src, tabs[2], tabs[3], bins)
            for a_, b_, name in zip(again, first, GRAD_NAMES):
                assert torch.equal(a_, b_), (src.dtype, name)
    live = sq.cuda()                      # the forward writes only the live square of each graph
    for _ in range(3):
        assert torch.equal(ops.bias_fwd_raw(pk, *tabs, out_dtype=torch.bfloat16)[live], f0[live])


# ---------------------------------------------------------------------------------------------------------------- GPU: K3
def _batch(sizes, seed=60):
    from mobgt_b200 import collator, synth
    w = synth.make_world("c1", seed=1)
    items = []
    for k, n in enumerate(sizes):
        items += synth.make_items(w, 1, 512, seed=seed + k, n_fixed=n, start=k)
    return collator.collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=1024, world=w)


def _bias(b, dtype=torch.bfloat16, seed=9):
    """the 12-head K2 forward on a collated batch"""
    from mobgt_b200 import ops
    from test_k2_k3_k4 import tables
    R, Pp, E, W, t = tables(H=H, seed=seed)
    cu = [x.cuda().contiguous() for x in (R, Pp, E, W.view(-1), t.view(-1))]
    return ops.bias_fwd_raw(b, *cu, out_dtype=dtype)


# <= 16 tokens (SIMT), 17..128, 129, 130..257 and 513 tokens; 12 heads give more than 296 (graph, head) items
MIXED = [3, 9, 15, 16, 60, 127, 128, 129, 200, 256, 512] + [16 + (7 * k) % 45 for k in range(20)]
SMALL_BOX = [1, 7, 15, 16, 40, 100, 127, 128, 128, 64]


def _ref64(qkv, bias, tok_off, drop=None):
    """float64 attention at 12 heads x 16 (out, lse), differentiable in qkv and bias"""
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
def test_h12_attention_batch_covers_every_path(lib_built):
    b = _batch(MIXED)
    t = np.diff(b.tok_off.cpu().numpy())
    assert t.min() <= 16 and ((t > 16) & (t <= 128)).any() and (t == 129).any() and ((t >= 130) & (t <= 257)).any()
    assert (t == 513).any() and int((t > 16).sum()) * H > 296


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.1])
def test_h12_attention_fwd_bwd_all_modes_match_float64(lib_built, p):
    """out / lse and dq / dk / dv / dS (modes 0, 1, 2) at 12 heads against float64 autograd with the same dropout mask; mode 1
    adds exactly dS, mode 2 is mode 0's dS rounded once to bf16, all three give the same dqkv."""
    from mobgt_b200 import ops
    b = _batch(MIXED, seed=80)
    bias = _bias(b, seed=4)
    assert bias.shape[1] == H
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
    ref, ref_lse = _ref64(q64, b64, tok_off, drop=(p, seed) if p > 0 else None)
    assert out.shape == (ntok, H * D16)
    assert (out.double().cpu() - ref.detach()).abs().max().item() <= 2e-2 * max(1.0, ref.abs().max().item())
    assert (lse.double().cpu() - ref_lse.detach()).abs().max().item() <= 2e-2
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
def test_h12_single_box_and_general_backward_agree(lib_built):
    """All graphs <= 129 tokens: mode 2 takes the single-box backward, mode 0 the general one; within 1e-2 of the gradient's
    magnitude of each other and 2e-2 of float64."""
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
def test_h12_attention_f32_kernels_match_torch(lib_built):
    """mobgt_attn_f32_fwd_hd / _bwd_hd at 12 heads x 16, T = 2 .. 301: within 1e-5 of torch fp32 autograd, with and without
    dropout; bitwise reproducible."""
    from mobgt_b200 import ops
    from test_k2_k3_k4 import torch_attention_diff
    TOL = 1e-5
    b = _batch((1, 3, 7, 15, 16, 40, 127, 128, 129, 200, 256, 300), seed=170)
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
MODEL_CASES = {
    "toyota": ("toyotagraph", [(2, 1, 512, 51), (None, 6, 40, 52), (128, 1, 512, 53), (300, 1, 512, 54)]),
    "gowalla": ("gowalla_nevda", [(2, 1, 512, 61), (None, 6, 40, 62), (129, 1, 512, 63), (300, 1, 512, 64)]),
}


def _pair(dataset_name, spec, seed=3, precision=16, num_heads=12):
    """oracle + product model at (num_heads, 128) with the same weights, and the two batches of the same items"""
    from mobgt_b200 import collator, model, synth
    w = synth.make_world("c1", seed=seed, dataset_name=dataset_name)
    items = []
    for n_fixed, cnt, cap, sd in spec:
        items += synth.make_items(w, cnt, cap, seed=sd, n_fixed=n_fixed, start=len(items))
    torch.manual_seed(seed)
    om = mo.Graphormer(w, n_layers=2, num_heads=num_heads, hidden_dim=128, ffn_dim=256, dataset_name=dataset_name).eval()
    with torch.no_grad():
        for emb in (om.edge_encoder, om.rel_pos_encoder, om.poi_pos_encoder):
            emb.weight.mul_(0.3)
            emb.weight[0].zero_()
        om.edge_dis_encoder.weight.mul_(0.3)
    pm = model.Graphormer(dataset_name=dataset_name, world=w, precision=precision, **_hp(num_heads)).cuda().eval()
    missing, _ = pm.load_state_dict(om.state_dict(), strict=False)
    assert not missing, missing
    assert pm.edge_encoder.weight.shape[1] == num_heads
    ob = mo.collate([mo.preprocess_item(it, hop_cap=20) for it in items], w, multi_hop_max_dist=20, rel_pos_max=1024)
    pb = collator.collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=1024, world=w)
    assert pb.N == 300 and min(pb.n_host) <= 15
    return om, pm, ob, pb


def _train_mode(*ms):
    for m_ in ms:
        m_.train()
        m_.poi_distance_model.eval()
        m_.poi_cat_model.eval()


def _fp32_errors(case, num_heads):
    """precision=32 model against the oracle: logits and loss within 1e-5; returns {parameter: (error vs the fp32 oracle,
    error vs the oracle run in float64)}, norm-wise"""
    from test_fp32_mode import _oracle_float64
    TOL = 1e-5
    om, pm, ob, pb = _pair(*MODEL_CASES[case], precision=32, num_heads=num_heads)
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
        if r.abs().max().item() < 1e-6 * gmax:
            assert g.abs().max().item() < 1e-4 * gmax, k
            continue
        r64 = ref64_g[k]
        table[k] = ((g - r).norm().item() / r.norm().item(), (g.double() - r64).norm().item() / r64.norm().item())
    return table


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(MODEL_CASES))
def test_12_heads_fp32_mode_matches_oracle(lib_built, case):
    """precision=32 at (12, 128): logits and loss within 1e-5; every parameter gradient within 1e-5 norm-wise of the fp32
    oracle or of its float64 run (test_fp32_mode.py's gate).  A gradient that misses both must be no further from float64 than
    2.5x the canonical 8-head model's gradient on the same items (the edge tables on a batch with a 300-node graph: K2's fp32
    histogram sums of nearly cancelling dS, see test_head_dim16.test_hidden64_fp32_mode_matches_oracle)."""
    from mobgt_b200 import model
    TOL = 1e-5
    try:
        table = _fp32_errors(case, 12)
        assert len(table) > 40
        miss = {k: e for k, e in table.items() if min(e) > TOL}
        if miss:
            print("12-head fp32 gradients outside 1e-5 (vs fp32 oracle, vs float64):", miss)
            canon = _fp32_errors(case, 8)
            worse = {k: (e, canon.get(k)) for k, e in miss.items() if k not in canon or e[1] > 2.5 * max(canon[k][1], TOL)}
            assert not worse, worse
    finally:
        model.ops.enable_tf32(True)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(MODEL_CASES))
def test_12_heads_bf16_mode_matches_oracle(lib_built, case):
    """precision=16 at (12, 128): logits and loss within 2e-2; every parameter gradient within 2e-2 norm-wise, or no worse than
    2.5x the error of the oracle under torch.autocast(bfloat16) (test_round2_gpu.test_canonical_model_on_baseline_shapes)."""
    from test_round2_gpu import _grad_table
    om, pm, ob, pb = _pair(*MODEL_CASES[case])
    with torch.no_grad():
        ref = om(ob)
        got = pm(pb)
    for a, r in zip(got, ref):
        assert a.shape == r.shape
        assert (a.float().cpu() - r).abs().max().item() <= 2e-2 * max(1.0, r.abs().max().item())
    om16 = copy.deepcopy(om)
    gcn16 = om16.gcn_tables

    def gcn_fp32():
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
@pytest.mark.parametrize("precision", [16, 32])
def test_12_heads_entry_trains_and_tests(lib_built, precision, tmp_path):
    """`entry --num_heads 12 --hidden_dim 128`: five training steps (precision 16: CUDA-graph replays of the bucketed step), a
    finite loss, then `--test` on the checkpoint returns the metric dict."""
    from mobgt_b200 import entry, model
    common = ["--dataset_name", "toyotagraph", "--gpus", "1", "--precision", str(precision), "--batch_size", "16",
              "--hidden_dim", "128", "--num_heads", "12", "--n_layers", "2", "--ffn_dim", "256", "--dropout_rate", "0.1",
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
