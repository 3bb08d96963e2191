"""The direct edge encoding: `Graphormer(edge_type=<anything but "multi_hop">)` (Graphormer's else-branch: the edge term of a pair
is edge_encoder[attn_edge_type], no walk, no edge_dis_encoder, no division by the distance).

CPU: the constructor accepts the mode at every supported shape, the head-count and argument checks of the new K2 entry points,
and a float64 reference `k2_direct_reference` pinned to `DirectOracle` (the oracle model of oracle/model_oracle.py with
Graphormer's else-branch in its bias build) at 8 and 12 heads.
GPU: the direct K2 kernels (forward fp32 / bf16, backward from one fp32 plane or 1 / 6 / 7 bf16 layer planes) against that
reference on packed batches whose feat8 plane is all zero, trajectory-like or dense random (tolerances of
tests/test_k2_bias_adversarial.py), the whole model in both precisions against `DirectOracle`, and
`entry --edge_type single_hop`."""
import copy
import ctypes
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import model_oracle as mo
from test_k2_bias_adversarial import SMALLS, _chain_item, live_mask, pair_index
from test_num_heads12 import MODEL_CASES, _hp, _train_mode

NEG_INF = float("-inf")
SHAPES = [(8, 128), (8, 64), (12, 128)]


# ---------------------------------------------------------------------------------------------------------------- reference
class DirectOracle(mo.Graphormer):
    """The oracle model with Graphormer's direct edge encoding in place of the multi-hop block of attn_bias_build: the
    reference's else-branch between model_fqandtoyo.py:1168-1208 and the add at :1213-1216,
        edge_input = self.edge_encoder(attn_edge_type).mean(-2).permute(0, 3, 1, 2)
    The rest of the bias (:1143-1165, :1216) is restated from mo.Graphormer.attn_bias_build.  The collator pads
    attn_edge_type to n_node + 1 rows and columns with the nodes first, so the node block is its leading [n_node, n_node]
    corner.  `mode` is ignored: the reference's fp16 round trips ('ref_half') belong to the multi-hop bmm."""

    def attn_bias_build(self, b, mode="fp32"):
        H = self.num_heads
        attn_bias, rel_pos, poi_pos = b.attn_bias, b.rel_pos, b.poi_pos
        n_node = b.x.size(1)
        g = attn_bias.clone().unsqueeze(1).repeat(1, H, 1, 1)                                # :1143-1147
        g[:, :, 1:, 1:] = g[:, :, 1:, 1:] + self.rel_pos_encoder(rel_pos).permute(0, 3, 1, 2) \
            + self.poi_pos_encoder(poi_pos).permute(0, 3, 1, 2)                                 # :1151-1158
        t = self.graph_token_virtual_distance.weight.view(1, H, 1).unsqueeze(-2)
        g[:, :, 1:, :1] = g[:, :, 1:, :1] + t                                                 # :1160-1165
        e = self.edge_encoder(b.attn_edge_type[:, :n_node, :n_node]).mean(-2).permute(0, 3, 1, 2)
        g[:, :, 1:, 1:] = g[:, :, 1:, 1:] + e                                                 # :1213-1215
        return g + attn_bias.unsqueeze(1)                                                     # :1216


def k2_direct_reference(n, rel_pos, poi_pos, feat, rel_pos_max, R, Ppos, E, tvd):
    """Dense bias [B, H, T, T] (H = R.shape[1], T = max n_g + 1) in the tables' dtype from packed per-pair indices (rel_pos,
    poi_pos, feat [cells]).  Row 0 is 0; column 0 of rows 1..n_g is tvd; cell (a, b) with a, b >= 1 is
    R[rp] + Ppos[pp] + E[f] with the indices of pair (a - 1, b - 1), -inf where rp - 1 >= rel_pos_max.  Cells outside a
    graph's (n_g + 1)^2 square are 0.  Differentiable in the four tables."""
    n = [int(v) for v in n]
    nh = R.shape[1]
    B, T = len(n), max(n) + 1
    rp, pp, f = (torch.as_tensor(x).long() for x in (rel_pos, poi_pos, feat))
    val = R[rp] + Ppos[pp] + E[f]
    val = torch.where(((rp - 1) >= rel_pos_max)[:, None], torch.full_like(val, NEG_INF), val)
    g, i, j = pair_index(n)
    out = torch.zeros(B, nh, T, T, dtype=R.dtype)
    out[g, :, i + 1, j + 1] = val
    for gi, k in enumerate(n):
        out[gi, :, 1:k + 1, 0] = tvd.reshape(nh, 1)
    return out


def _tables(H, bins, seed, scale=0.3):
    """R, Ppos, E, tvd in float64.  E row 0 is NOT zero: the direct encoding reads it for every pair without an edge."""
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(r, H, generator=g, dtype=torch.float64) * scale for r in (512, bins, 128)] + \
        [torch.randn(H, generator=g, dtype=torch.float64) * scale]


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("num_heads,hidden_dim", SHAPES)
@pytest.mark.parametrize("edge_type", ["single_hop", "no such encoding"])
def test_constructor_accepts_direct_edge_types(num_heads, hidden_dim, edge_type):
    from mobgt_b200 import model, synth
    w = synth.make_world("tiny", seed=1)
    m = model.Graphormer(dataset_name="toyotagraph", world=w, **_hp(num_heads, hidden_dim, edge_type=edge_type))
    assert m.direct_edges and m.edge_type == edge_type
    ref = model.Graphormer(dataset_name="toyotagraph", world=w, **_hp(num_heads, hidden_dim))
    assert not ref.direct_edges
    assert list(m.state_dict()) == list(ref.state_dict())          # edge_dis_encoder is kept in both modes
    assert m.edge_dis_encoder.weight.shape == (128 * num_heads * num_heads, 1)


@pytest.mark.parametrize("num_heads,hidden_dim", [(12, 64), (16, 192), (4, 128)])
def test_constructor_still_rejects_unsupported_shapes_in_direct_mode(num_heads, hidden_dim):
    from mobgt_b200 import model, synth
    w = synth.make_world("tiny", seed=1)
    with pytest.raises(NotImplementedError) as e:
        model.Graphormer(dataset_name="toyotagraph", world=w, **_hp(num_heads, hidden_dim, edge_type="single_hop"))
    assert "(12, 128)" in str(e.value)


def test_direct_entry_points_reject_unbuilt_head_counts_and_bad_arguments(lib_built):
    """num_heads is checked before anything else: 4, 16 and 32 return MOBGT_ERR_UNSUPPORTED (-3) naming 8 and 12.  The
    workspace query returns < 0 on a bad head count, T or num_bins."""
    from mobgt_b200 import _C
    L = _C.lib()
    for nh in (4, 16, 32):
        for name in ("mobgt_bias_direct_fwd", "mobgt_bias_direct_bwd"):
            argt = _C.SIGNATURES[name]
            args = [None if t is ctypes.c_void_p else 0 for t in argt]
            args[8] = nh                                      # (n, sq_off, rel_pos, poi_pos, feat, B, T, Tp, H, ...)
            assert getattr(L, name)(*args) == -3, (name, nh)
            assert "8 and 12" in _C.last_error(), (name, _C.last_error())
        assert L.mobgt_bias_direct_bwd_workspace_bytes(129, 64, nh) < 0
    for H in (8, 12):
        for T, bins in ((1, 64), (129, 0), (129, 1025), (0, 1)):
            assert L.mobgt_bias_direct_bwd_workspace_bytes(T, bins, H) < 0, (T, bins, H)
        for T, bins in ((2, 1), (129, 64), (513, 1024)):
            assert L.mobgt_bias_direct_bwd_workspace_bytes(T, bins, H) > 0
        # null pointers and bad shapes return a status
        argt = _C.SIGNATURES["mobgt_bias_direct_fwd"]
        args = [None if t is ctypes.c_void_p else 1 for t in argt]
        args[8] = H
        assert L.mobgt_bias_direct_fwd(*args) == -6 and "null" in _C.last_error()


def _packed_direct_from_oracle(ob):
    n = (ob.x[:, :, 0] != 0).sum(1).tolist()
    rel, poi, feat = [], [], []
    for g, k in enumerate(n):
        rel.append(ob.rel_pos[g, :k, :k].reshape(-1))
        poi.append(ob.poi_pos[g, :k, :k].reshape(-1))
        feat.append(ob.attn_edge_type[g, :k, :k, 0].reshape(-1))
    return n, torch.cat(rel), torch.cat(poi), torch.cat(feat)


@pytest.mark.parametrize("H", [8, 12])
@pytest.mark.parametrize("rel_pos_max", [1024, 20, 3])
def test_direct_reference_equals_oracle_else_branch(H, rel_pos_max):
    """k2_direct_reference on the packed indices of an oracle-collated batch == DirectOracle.attn_bias_build run in float64:
    finite cells within 1e-12 of the cell's magnitude bound, identical -inf sets."""
    from mobgt_b200 import synth
    w = synth.make_world("c1", seed=1)
    items = synth.make_items(w, 5, 40, seed=H + rel_pos_max) + [_chain_item(w, 33, 7, 5), _chain_item(w, 4, 8, 6)]
    ob = mo.collate([mo.preprocess_item(it, hop_cap=20) for it in items], w, multi_hop_max_dist=20, rel_pos_max=rel_pos_max)
    R, Pp, E, t = _tables(H, w.num_bins, seed=rel_pos_max)
    m = DirectOracle.__new__(DirectOracle)
    torch.nn.Module.__init__(m)
    m.num_heads, m.multi_hop_max_dist = H, 20
    m.rel_pos_encoder = torch.nn.Embedding.from_pretrained(R.clone(), freeze=False, padding_idx=0)
    m.poi_pos_encoder = torch.nn.Embedding.from_pretrained(Pp.clone(), freeze=False, padding_idx=0)
    m.edge_encoder = torch.nn.Embedding.from_pretrained(E.clone(), freeze=False, padding_idx=0)
    m.graph_token_virtual_distance = torch.nn.Embedding.from_pretrained(t.view(1, -1).clone(), freeze=False)
    ob64 = copy.copy(ob)
    ob64.attn_bias = ob.attn_bias.double()
    with torch.no_grad():
        orc = m.attn_bias_build(ob64, "fp32")
    assert orc.dtype == torch.float64
    n, rel, poi, feat = _packed_direct_from_oracle(ob)
    assert (feat != 0).any() and (feat == 0).any()
    ref = k2_direct_reference(n, rel, poi, feat, rel_pos_max, R, Pp, E, t)
    A = k2_direct_reference(n, rel, poi, feat, rel_pos_max, R.abs(), Pp.abs(), E.abs(), t.abs())
    T = max(n) + 1
    assert orc.shape == ref.shape == (len(n), H, T, T)
    live = live_mask(n, T).expand_as(ref)
    o, r, a = orc[live], ref[live], A[live]
    assert torch.equal(torch.isneginf(o), torch.isneginf(r))
    fin = torch.isfinite(r)
    assert ((o[fin] - r[fin]).abs() <= 1e-12 * a[fin]).all()
    if rel_pos_max < 1024:
        assert torch.isneginf(r).any() and fin.any()


# ------------------------------------------------------------------------------------------------ packed batches (GPU)
def direct_batch(seed, ns, num_bins, rel_pos_max, pattern):
    """Packed inputs of the direct K2 kernels for graphs of ns nodes.  rel_pos: 1 on the diagonal, elsewhere a mix of 0 / 1,
    2..n_g, n_g+1..510 (keys >= T lie past the backward's histogram plan) and 511.  feat8: "zero" (no edges), "traj" (a few
    3s and 4s per row, diagonal 0) or "dense" (uniform 0..127, diagonal included)."""
    rng = np.random.default_rng(seed)
    rels, pois, feats = [], [], []
    for n in ns:
        C = n * n
        i, j = np.repeat(np.arange(n), n), np.tile(np.arange(n), n)
        cat = rng.choice(4, size=C, p=[0.06, 0.34, 0.34, 0.26])
        key = np.select([cat == 0, cat == 1, cat == 2],
                        [rng.integers(0, 2, C), rng.integers(2, min(max(n, 2), 510) + 1, C),
                         rng.integers(n + 1, 511, C) if n < 510 else rng.integers(2, 511, C)], 511)
        key = np.where(i == j, 1, key)
        if pattern == "zero":
            f = np.zeros(C, np.int64)
        elif pattern == "traj":
            f = np.where(rng.random(C) < min(1.0, 3.0 / n), rng.choice([3, 4], size=C), 0)
            f = np.where(i == j, 0, f)
        else:
            f = rng.integers(0, 128, C)
        rels.append(key)
        pois.append(rng.integers(0, num_bins, C))
        feats.append(f)
    n = np.asarray(ns, np.int32)
    sq = np.zeros(len(ns) + 1, np.int64)
    np.cumsum(n.astype(np.int64) ** 2, out=sq[1:])
    h_rel = torch.from_numpy(np.concatenate(rels).astype(np.int16))
    h_poi = torch.from_numpy(np.concatenate(pois).astype(np.int16))
    h_feat = torch.from_numpy(np.concatenate(feats).astype(np.uint8))
    return SimpleNamespace(B=len(ns), N=int(n.max()), n=torch.from_numpy(n).cuda(), n_host=n, sq_off=torch.from_numpy(sq).cuda(),
                           rel_pos16=h_rel.cuda(), poi_pos16=h_poi.cuda(), feat8=h_feat.cuda(), rel_pos_max=rel_pos_max,
                           h_rel=h_rel.long(), h_poi=h_poi.long(), h_feat=h_feat.long())


# (H, graph sizes, num_bins, rel_pos_max, extra pitch, bf16 layer planes, feat8 pattern); T = max n + 1 covers every residue mod 8
DIRECT_CASES = [
    (8, [1], 64, 1024, 0, 1, "dense"),                  # T = 2
    (12, [2, 3, 1, 3], 1, 20, 0, 6, "traj"),            # T = 4
    (8, [12, 5, 1, 9], 1024, 3, 0, 7, "dense"),         # T = 13
    (12, [13, 2, 7], 64, 1024, 0, 1, "zero"),           # T = 14
    (8, [14, 14, 3], 1, 1024, 0, 6, "traj"),            # T = 15
    (12, [15, 8, 1], 1024, 20, 0, 7, "dense"),          # T = 16
    (8, [16, 4, 11, 16], 64, 3, 0, 1, "traj"),          # T = 17
    (12, [17, 2], 64, 1024, 24, 6, "dense"),            # T = 18, pitch 48 > round_up(T, 8)
    (8, [35, 20, 6], 64, 20, 0, 7, "zero"),             # T = 36
    (12, [130, 64, 3], 1024, 1024, 0, 1, "traj"),       # T = 131
    (8, [200, 1, 2], 1, 1024, 0, 6, "dense"),           # T = 201
    (12, [299, 150, 40, 7], 64, 1024, 0, 7, "traj"),    # T = 300
    (8, [509, 12], 64, 20, 0, 1, "traj"),               # T = 510: key 510 is the only one past the plan
    (12, [512] + SMALLS, 1024, 1024, 0, 6, "dense"),    # T = 513
    (8, [512] + SMALLS, 64, 3, 0, 7, "traj"),           # T = 513
    (12, [47, 3, 3], 1024, 1024, 0, 7, "zero"),         # T = 48
]


def _case_id(c):
    return f"H{c[0]}-T{max(c[1]) + 1}-bins{c[2]}-rpm{c[3]}-{c[6]}"


def test_direct_case_matrix():
    assert {(max(c[1]) + 1) % 8 for c in DIRECT_CASES} == set(range(8))
    assert {c[0] for c in DIRECT_CASES} == {8, 12} and {c[2] for c in DIRECT_CASES} == {1, 64, 1024}
    assert {c[3] for c in DIRECT_CASES} == {1024, 20, 3} and {c[6] for c in DIRECT_CASES} == {"zero", "traj", "dense"}
    assert {1, 6, 7} <= {c[5] for c in DIRECT_CASES} and any(c[4] for c in DIRECT_CASES)


def _reference_grads(pk, tabs, dB):
    """Gradients of sum(bias * dB) over the finite cells w.r.t. (R, Ppos, E, tvd), float64 autograd."""
    leaves = [t.detach().double().clone().requires_grad_(True) for t in tabs]
    out = k2_direct_reference(pk.n_host, pk.h_rel, pk.h_poi, pk.h_feat, pk.rel_pos_max, *leaves)
    fin = torch.isfinite(out)
    (torch.where(fin, out, torch.zeros_like(out)) * dB).sum().backward()
    return [lf.grad for lf in leaves]


GRAD_NAMES = ("dR", "dPpos", "dE", "dtvd")


def _check_grads(got, ref, A, tag):
    """|got - ref| <= 2e-5 * A_entry; dE row 0 (the padding row) is exactly 0 and rows 1.. are checked."""
    for name, g, r, a in zip(GRAD_NAMES, got, ref, A):
        g = g.detach().double().cpu().reshape(r.shape)
        if name == "dE":
            assert (g[0] == 0).all(), tag
            g, r, a = g[1:], r[1:], a[1:]
        if name == "dR":                  # padding_idx row 0 is zeroed by the autograd nodes, not by the kernel
            g, r, a = g[1:], r[1:], a[1:]
        err = (g - r).abs()
        bad = err > 2e-5 * a
        assert not bad.any(), (tag, name, int(bad.sum()), float(err.max()))


def _bwd_strided(pk, flat, n_layers, ls, T, Tp, H, bins):
    """mobgt_bias_direct_bwd with bf16 planes ls elements apart"""
    from mobgt_b200 import _C
    dev = flat.device
    ws_bytes = int(_C.lib().mobgt_bias_direct_bwd_workspace_bytes(T, bins, H))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    out = [torch.empty(r, H, device=dev) for r in (512, bins, 128)] + [torch.empty(H, device=dev)]
    _C.call("mobgt_bias_direct_bwd", _C.ptr(pk.n), _C.ptr(pk.sq_off), _C.ptr(pk.rel_pos16), _C.ptr(pk.poi_pos16),
            _C.ptr(pk.feat8), pk.B, T, Tp, H, pk.rel_pos_max, bins, flat.data_ptr(), 1, n_layers, ls, _C.ptr(ws), ws_bytes,
            *[_C.ptr(x) for x in out], _C.stream_ptr())
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("case", DIRECT_CASES, ids=_case_id)
def test_k2_direct_fwd_bwd_matches_float64(lib_built, case):
    """mobgt_bias_direct_fwd (fp32 and bf16) and mobgt_bias_direct_bwd (one fp32 plane; n_layers bf16 planes, contiguous and
    further apart) against k2_direct_reference in float64: forward within 1e-5 * A_cell (bf16: plus 2^-8 |ref|), -inf exactly
    where rel_pos_max masks; dR, dPpos, dE, dtvd within 2e-5 * A_entry, dE row 0 exactly 0; three repeats bitwise equal; NaN in
    dBias cells the kernel must not read changes no bit."""
    from mobgt_b200 import ops
    H, ns, bins, rpm, extra, n_layers, pattern = case
    seed = 7 * sum(ns) + H + bins
    pk = direct_batch(seed, ns, bins, rpm, pattern)
    T = pk.N + 1
    Tp = ops.bias_pitch(T) + extra
    if max(ns) > 20:
        assert (pk.h_rel == 511).any()
        if T < 511:                                                         # keys min(T, 511)..510: past the histogram plan
            assert ((pk.h_rel >= T) & (pk.h_rel < 511)).any()
    tabs = _tables(H, bins, seed)
    A_tabs = [x.abs() for x in tabs]
    ref = k2_direct_reference(pk.n_host, pk.h_rel, pk.h_poi, pk.h_feat, rpm, *tabs)
    A = k2_direct_reference(pk.n_host, pk.h_rel, pk.h_poi, pk.h_feat, rpm, *A_tabs)
    live = live_mask(pk.n_host, T).expand_as(ref)
    masked = torch.isneginf(ref) & live
    fin = live & ~masked
    cu = [x.float().cuda().contiguous() for x in tabs]
    for dt in (torch.float32, torch.bfloat16):
        out = ops.bias_direct_fwd_raw(pk, *cu, out_dtype=dt, T=T, Tp=Tp)
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
    used = torch.zeros(pk.B, H, T, Tp, dtype=torch.bool)
    used[..., :T] = fin
    used[:, :, 0, :] = False
    # ---- one fp32 plane
    dB = torch.where(sq, torch.randn(pk.B, H, T, Tp, generator=gen), torch.zeros(()))
    dB64 = dB[..., :T].double()
    got32 = ops.bias_direct_bwd_raw(pk, dB.cuda(), bins)
    _check_grads(got32, _reference_grads(pk, tabs, dB64), _reference_grads(pk, A_tabs, dB64.abs()), "f32")
    for _ in range(3):
        again = ops.bias_direct_bwd_raw(pk, dB.cuda(), bins)
        for a_, b_, name in zip(again, got32, GRAD_NAMES):
            assert torch.equal(a_, b_), ("f32 repeat", name)
    dirty = torch.where(used, dB, torch.full((), float("nan")))
    again = ops.bias_direct_bwd_raw(pk, dirty.cuda(), bins)
    for a_, b_, name in zip(again, got32, GRAD_NAMES):
        assert torch.equal(a_, b_), ("f32 NaN fill", name)
    # ---- n_layers bf16 planes, summed in the kernel
    planes = torch.stack([(torch.randn(pk.B, H, T, Tp, generator=gen) * (0.5 + 0.25 * l)).to(torch.bfloat16)
                          for l in range(n_layers)])
    planes = torch.where(sq.unsqueeze(0), planes, torch.zeros((), dtype=torch.bfloat16))
    psum = planes.double().sum(0)[..., :T]
    got16 = ops.bias_direct_bwd_raw(pk, planes.cuda(), bins)
    _check_grads(got16, _reference_grads(pk, tabs, psum), _reference_grads(pk, A_tabs, planes.double().abs().sum(0)[..., :T]),
                 f"bf16 x{n_layers}")
    for _ in range(3):
        again = ops.bias_direct_bwd_raw(pk, planes.cuda(), bins)
        for a_, b_, name in zip(again, got16, GRAD_NAMES):
            assert torch.equal(a_, b_), ("bf16 repeat", name)
    dirty16 = torch.where(used.unsqueeze(0), planes, torch.full((), float("nan"), dtype=torch.bfloat16))
    again = ops.bias_direct_bwd_raw(pk, dirty16.cuda(), bins)
    for a_, b_, name in zip(again, got16, GRAD_NAMES):
        assert torch.equal(a_, b_), ("bf16 NaN fill", name)
    plane = pk.B * H * T * Tp
    ls = plane + 40
    flat = torch.full((n_layers * ls,), float("nan"), dtype=torch.bfloat16)
    flat.view(n_layers, ls)[:, :plane] = dirty16.reshape(n_layers, plane)
    gs = _bwd_strided(pk, flat.cuda(), n_layers, ls, T, Tp, H, bins)
    for a_, b_, name in zip(gs, got16, GRAD_NAMES):
        assert torch.equal(a_, b_), ("bf16 strided", name)


# ---------------------------------------------------------------------------------------------------------------- GPU model
def _pair_direct(num_heads, precision, seed=3):
    """oracle + product model at (num_heads, 128), edge_type "single_hop", the same weights (edge_encoder row 0 nonzero), and
    the oracle-collated and packed batches of the same items (graphs of 2..300 nodes)."""
    from mobgt_b200 import collator, model, synth
    dataset_name, spec = MODEL_CASES["toyota"]
    w = synth.make_world("c1", seed=seed, dataset_name=dataset_name)
    items = []
    for n_fixed, cnt, cap, sd in spec:
        items += synth.make_items(w, cnt, cap, seed=sd, n_fixed=n_fixed, start=len(items))
    torch.manual_seed(seed)
    om = DirectOracle(w, n_layers=2, num_heads=num_heads, hidden_dim=128, ffn_dim=256, dataset_name=dataset_name).eval()
    with torch.no_grad():
        for emb in (om.edge_encoder, om.rel_pos_encoder, om.poi_pos_encoder):
            emb.weight.mul_(0.3)
        om.rel_pos_encoder.weight[0].zero_()
        om.poi_pos_encoder.weight[0].zero_()
        om.edge_encoder.weight[0].normal_(0.0, 0.3)
    pm = model.Graphormer(dataset_name=dataset_name, world=w, precision=precision,
                          **_hp(num_heads, edge_type="single_hop")).cuda().eval()
    missing, _ = pm.load_state_dict(om.state_dict(), strict=False)
    assert not missing, missing
    ob = mo.collate([mo.preprocess_item(it, hop_cap=20) for it in items], w, multi_hop_max_dist=20, rel_pos_max=1024)
    pb = collator.collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=1024, world=w)
    assert pb.N == 300 and (pb.feat8 != 0).any()
    return om, pm, ob, pb


def _grads(m, cpu=True):
    return {k: (p.grad.float().cpu() if cpu else p.grad) for k, p in m.named_parameters() if p.grad is not None}


@pytest.mark.gpu
@pytest.mark.parametrize("num_heads", [8, 12])
def test_direct_fp32_mode_matches_oracle(lib_built, num_heads):
    """precision=32, edge_type single_hop: logits (packed and reference-collated batch) and loss within 1e-5 of the fp32 oracle;
    every parameter gradient within 1e-5 norm-wise of the fp32 oracle or of its float64 run, or no further from float64 than
    2.5x the fp32 oracle itself is (test_k2_bias_adversarial's gate for sums of nearly cancelling dS); edge_dis_encoder's
    gradient exactly 0."""
    from mobgt_b200 import model
    from test_fp32_mode import _oracle_float64
    TOL = 1e-5
    try:
        om, pm, ob, pb = _pair_direct(num_heads, 32)
        with torch.no_grad():
            ref = om(ob)
            got = pm(pb)
            dense = pm(ob)
        for a, d, r in zip(got, dense, ref):
            assert a.dtype == torch.float32 and a.shape == r.shape
            assert (a.cpu() - r).abs().max().item() <= TOL * max(1.0, r.abs().max().item())
            assert (d.cpu() - a.cpu()).abs().max().item() <= 1e-6 * max(1.0, r.abs().max().item())
        _train_mode(om, pm)
        pm.pos_embed.p = 0.0
        lref = om.training_loss(ob)
        lref.backward()
        for p in pm.parameters():
            p.grad = torch.zeros_like(p)
        lgot = pm.training_step(pb)
        lgot.backward()
        assert abs(lgot.item() - lref.item()) <= TOL * abs(lref.item()), (lgot.item(), lref.item())
        assert not pm.edge_dis_encoder.weight.grad.any()
        ref_g, got_g = _grads(om, cpu=False), _grads(pm)
        _, ref64 = _oracle_float64(om, ob)
        gmax = max(r.abs().max().item() for r in ref_g.values())
        bad, checked = {}, 0
        for k, r in ref_g.items():
            g = got_g.get(k)
            if g is None or r.abs().max().item() < 1e-6 * gmax:
                assert g is None or g.abs().max().item() < 1e-4 * gmax, k
                continue
            checked += 1
            r64 = ref64[k]
            e32 = (g - r).norm().item() / r.norm().item()
            e64 = (g.double() - r64).norm().item() / r64.norm().item()
            o64 = (r.double() - r64).norm().item() / r64.norm().item()
            if min(e32, e64) > max(TOL, 2.5 * o64):
                bad[k] = (e32, e64, o64)
        assert checked > 40 and "edge_encoder.weight" in ref_g
        assert not bad, bad
    finally:
        model.ops.enable_tf32(True)


@pytest.mark.gpu
@pytest.mark.parametrize("num_heads", [8, 12])
def test_direct_bf16_mode_matches_oracle(lib_built, num_heads):
    """precision=16, edge_type single_hop: logits and loss within 2e-2; every parameter gradient within 2e-2 norm-wise, or no
    worse than 2.5x the error of the oracle under torch.autocast(bfloat16) (the gate of test_num_heads12); edge_dis_encoder's
    gradient exactly 0; the reference-collated batch gives the packed batch's logits."""
    from test_round2_gpu import _grad_table
    om, pm, ob, pb = _pair_direct(num_heads, 16)
    with torch.no_grad():
        ref = om(ob)
        got = pm(pb)
        dense = pm(ob)
    for a, d, r in zip(got, dense, ref):
        assert a.shape == r.shape
        assert (a.float().cpu() - r).abs().max().item() <= 2e-2 * max(1.0, r.abs().max().item())
        assert (d.float() - a.float()).abs().max().item() <= 1e-6 * max(1.0, r.abs().max().item())
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
    for p in pm.parameters():
        p.grad = torch.zeros_like(p)
    lgot = pm.training_step(pb)
    lgot.backward()
    assert abs(lgot.item() - lref.item()) <= 2e-2 * abs(lref.item()), (lgot.item(), lref.item())
    assert not pm.edge_dis_encoder.weight.grad.any()
    ref_g = _grads(om, cpu=False)
    ours = _grad_table(ref_g, _grads(pm))
    auto = _grad_table(ref_g, _grads(om16, cpu=False))
    assert len(ours) > 40 and "edge_encoder.weight" in ours
    bad = {k: (e, auto.get(k)) for k, e in ours.items() if e > max(2e-2, 2.5 * auto.get(k, 0.0))}
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("num_heads,hidden_dim", SHAPES)
def test_direct_entry_trains_validates_and_tests(lib_built, num_heads, hidden_dim, tmp_path):
    """`entry --edge_type single_hop` at each supported shape: five training steps with CUDA-graph replays and a finite loss,
    then `--validate` and `--test` on the checkpoint return finite metrics."""
    from mobgt_b200 import entry, model
    common = ["--dataset_name", "toyotagraph", "--gpus", "1", "--precision", "16", "--batch_size", "16",
              "--hidden_dim", str(hidden_dim), "--num_heads", str(num_heads), "--n_layers", "2", "--ffn_dim", "256",
              "--dropout_rate", "0.1", "--intput_dropout_rate", "0.1", "--attention_dropout_rate", "0.1", "--weight_decay", "0.0",
              "--peak_lr", "2e-4", "--end_lr", "1e-9", "--edge_type", "single_hop", "--warmup_updates", "40000",
              "--tot_updates", "400000", "--seed", "1", "--max_epochs", "1", "--synthetic", "tiny", "--train_graphs", "96",
              "--test_graphs", "24", "--multi_hop_max_dist", "20", "--default_root_dir", str(tmp_path)]
    try:
        r = entry.cli_main(common + ["--limit_train_steps", "5"])
        assert r["steps"] == 5 and np.isfinite(r["loss"]) and r["graph_steps"] >= 1, r
        ck = [os.path.join(dp, f) for dp, _, fs in os.walk(tmp_path) for f in fs if f == "last.ckpt"]
        assert len(ck) == 1
        for flag in ("--validate", "--test"):
            t = entry.cli_main(common + [flag, "--resume_from_checkpoint", ck[0]])
            m = t["metrics"]
            assert all(np.isfinite(m[k_]) for k_ in ("acc1", "acc5", "acc10", "acc20", "mrr")), (flag, m)
    finally:
        model.ops.enable_tf32(True)
