"""K2 (csrc/k2_bias.cu, attention-bias build forward / backward) against a float64 reference evaluated straight from the packed
indices, on inputs the collator of trajectory graphs rarely or never produces: walk bytes that deviate from the walk the distance
predicts (one, two, three or all of them, features below and above 16, walks cut short or longer than predicted), rel_pos keys
over the whole 0..511 range (keys past the backward's histogram plan included), every hop width, num_bins 1 / 64 / 1024 (every
backward warp plan from 1 to 12) and rel_pos_max 1024 / 20 / 3.  Then the rel_pos_max -inf mask through the attention kernels
(K3, tensor-core and SIMT, bf16 and fp32, with and without dropout) and through the whole model.

The reference (`k2_reference`) is pinned to the oracle's attn_bias_build (oracle/model_oracle.py) on oracle-collated batches by a
CPU test, so the GPU tests inherit the oracle's authority.  Tolerances are relative to magnitude bounds: the same functions
evaluated on |tables| and |dBias| give, per output element, the sum of the absolute values of the terms it is made of
(A_cell for the forward, A_entry for the backward).  A comparison against them can neither pass by cancellation nor fail by it."""
import copy
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import model_oracle as mo
from helpers import attn_drop_keep

H = 8
NEG_INF = float("-inf")


# ------------------------------------------------------------------------------------------------------------ reference
def pair_index(n):
    """(graph, i, j) of every packed pair, in the packed order (graph-major, then row-major over the n_g x n_g pairs)."""
    g = np.concatenate([np.full(k * k, gi) for gi, k in enumerate(n)]).astype(np.int64)
    i = np.concatenate([np.repeat(np.arange(k), k) for k in n]).astype(np.int64)
    j = np.concatenate([np.tile(np.arange(k), k) for k in n]).astype(np.int64)
    return torch.from_numpy(g), torch.from_numpy(i), torch.from_numpy(j)


def expected_walk(rp, dk):
    """Walk length the distance key rp = M + 1 predicts: min(M, dk) for a reachable pair (M < 510), else 0."""
    m = np.asarray(rp) - 1
    return np.where(m < 510, np.clip(m, 0, dk), 0)


def k2_reference(n, rel_pos, poi_pos, edge_in, dk, rel_pos_max, R, Ppos, E, W, tvd):
    """Dense bias [B, 8, T, T] (T = max n_g + 1) in the tables' dtype, from packed per-pair indices (rel_pos, poi_pos [cells],
    edge_in [cells, >= dk]).  Row 0 is 0; column 0 of rows 1..n_g is tvd; cell (a, b) with a, b >= 1 is
        R[rp] + Ppos[pp] + (sum_{k < dk} E[e_k] @ W[k]) / clamp(rp - 1, 1, dk)
    with rp, pp, e the indices of pair (a - 1, b - 1), and -inf where rp - 1 >= rel_pos_max.  Cells outside a graph's
    (n_g + 1)^2 square are 0.  Differentiable in the five tables."""
    n = [int(v) for v in n]
    B, T = len(n), max(n) + 1
    rp, pp, ei = (torch.as_tensor(x).long() for x in (rel_pos, poi_pos, edge_in))
    W3 = W.reshape(-1, H, H)
    e = torch.zeros(rp.numel(), H, dtype=R.dtype)
    for k in range(dk):
        e = e + (E @ W3[k])[ei[:, k]]            # == E[e_k] @ W[k], gathered after the product
    sp = (rp - 1).clamp(1, dk).to(R.dtype)
    val = R[rp] + Ppos[pp] + e / sp[:, None]
    val = torch.where(((rp - 1) >= rel_pos_max)[:, None], torch.full_like(val, NEG_INF), val)
    g, i, j = pair_index(n)
    out = torch.zeros(B, H, T, T, dtype=R.dtype)
    out[g, :, i + 1, j + 1] = val
    for gi, k in enumerate(n):
        out[gi, :, 1:k + 1, 0] = tvd.reshape(H, 1)
    return out


def live_mask(n, T, Tp=None):
    """bool [B, 1, T, Tp]: the (n_g + 1)^2 square of each graph."""
    Tp = Tp or T
    r = torch.arange(T).view(1, 1, T, 1)
    c = torch.arange(Tp).view(1, 1, 1, Tp)
    nn_ = torch.as_tensor(np.asarray(n)).view(-1, 1, 1, 1)
    return (r <= nn_) & (c <= nn_)


def reference_grads(pk, tabs, dB):
    """Gradients of sum(bias * dB) over the finite cells w.r.t. (R, Ppos, E, W, tvd), float64 autograd through k2_reference."""
    leaves = [t.detach().double().clone().requires_grad_(True) for t in tabs]
    out = k2_reference(pk.n_host, pk.h_rel, pk.h_poi, pk.h_edge, pk.dk, pk.rel_pos_max, *leaves)
    fin = torch.isfinite(out)
    (torch.where(fin, out, torch.zeros_like(out)) * dB).sum().backward()
    return [lf.grad for lf in leaves]


# --------------------------------------------------------------------------------------------------- CPU pin to the oracle
def _chain_item(world, n, seed, idx):
    """A trajectory of n distinct POIs visited once each: a directed chain, so M(i, j) = j - i for j > i and unreachable
    otherwise; long chains make every distance up to n - 1 occur."""
    from mobgt_b200 import synth
    rng = np.random.default_rng(seed)
    names = (rng.choice(world.P, size=n, replace=False) + 1).astype(np.int64)
    src = np.arange(n - 1, dtype=np.int64)
    slot = rng.integers(0, 48, size=n).astype(np.int64)
    return synth.Data(idx=idx, x=names.reshape(-1, 1), edge_index=np.stack([src, src + 1]),
                      edge_attr=np.ones(n - 1, np.int64), y=np.array([int(rng.integers(1, world.P + 1))], np.int64),
                      time=slot.reshape(-1, 1), time_normal=(slot / 48.0).astype(np.float32).reshape(-1, 1),
                      user=np.array([[int(rng.integers(0, world.U))]], np.int64), cat=world.cat_of_poi[names - 1].reshape(-1, 1))


def _tables(bins, hops, seed, scale=0.3):
    g = torch.Generator().manual_seed(seed)
    R = torch.randn(512, H, generator=g, dtype=torch.float64) * scale
    Pp = torch.randn(bins, H, generator=g, dtype=torch.float64) * scale
    E = torch.randn(128, H, generator=g, dtype=torch.float64) * scale
    W = torch.randn(hops * H * H, generator=g, dtype=torch.float64) * scale
    t = torch.randn(H, generator=g, dtype=torch.float64) * scale
    E[0] = 0                      # edge_encoder row 0 is the padding row (nn.Embedding(padding_idx=0)): part of K2's domain
    return R, Pp, E, W, t


def _packed_from_oracle(ob, dk):
    n = (ob.x[:, :, 0] != 0).sum(1).tolist()
    hops = (dk + 3) // 4 * 4
    rel, poi, edge = [], [], []
    for g, k in enumerate(n):
        rel.append(ob.rel_pos[g, :k, :k].reshape(-1))
        poi.append(ob.poi_pos[g, :k, :k].reshape(-1))
        e = ob.edge_input[g, :k, :k, :, 0].reshape(k * k, -1)
        edge.append(torch.nn.functional.pad(e, (0, hops - e.shape[1])))
    return n, torch.cat(rel), torch.cat(poi), torch.cat(edge)


@pytest.mark.parametrize("rel_pos_max", [1024, 20, 3])
@pytest.mark.parametrize("dk", [5, 20])
def test_reference_equals_oracle_attn_bias_build(rel_pos_max, dk):
    """k2_reference on the packed indices of an oracle-collated batch == model_oracle.Graphormer.attn_bias_build run in float64
    on that batch: finite cells within 1e-12 of the cell's magnitude bound, identical -inf sets (CPU only)."""
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
    ref = k2_reference(n, rel, poi, edge, dk, rel_pos_max, R, Pp, E, W, t)
    A = k2_reference(n, rel, poi, edge, dk, rel_pos_max, R.abs(), Pp.abs(), E.abs(), W.abs(), t.abs())
    T = max(n) + 1
    assert orc.shape == ref.shape == (len(n), H, T, T)
    live = live_mask(n, T).expand_as(ref)
    o, r, a = orc[live], ref[live], A[live]
    assert torch.equal(torch.isneginf(o), torch.isneginf(r))
    assert torch.isfinite(r[~torch.isneginf(r)]).all()
    fin = torch.isfinite(r)
    assert ((o[fin] - r[fin]).abs() <= 1e-12 * a[fin]).all()
    if rel_pos_max < 1024:
        assert torch.isneginf(r).any() and fin.any()


# ------------------------------------------------------------------------------------------------ adversarial packed batches
def k2_bwd_plan(T, hops, num_bins):
    """Python restatement of k2_bwd_plan (csrc/k2_bias.cu): (histogram rows, partial-row stride, warps per CTA)."""
    rrows = min(T, 511) + 1
    nR, nP = rrows * H, num_bins * H
    stride = hops * 16 * H + nR + nP + H
    pitch = ((((T + 3) & ~3) + 27) // 32) * 32 + 4
    per_warp = 2 * (nR + H) + 2 * (nP + H) + H * pitch + 3 * pitch + H
    cta_words = (hops + 1) * 8 + 40
    return rrows, stride, min((227 * 1024 - 2048 - cta_words * 4) // (per_warp * 4), 12)


def _features(rng, size):
    """edge features: half from 1..15 (the backward's per-CTA table), half from 16..127 (its launch-wide table)"""
    small = rng.random(size) < 0.5
    return np.where(small, rng.integers(1, 16, size), rng.integers(16, 128, size)).astype(np.int64)


def adversarial_batch(seed, ns, hops, dk, num_bins, rel_pos_max):
    """Packed K2 inputs (what ops.bias_fwd_raw / bias_bwd_raw read) for graphs of ns nodes, inside K2's input domain
    (include/mobgt.h) but far from trajectory-graph statistics.  Per pair:
      rel_pos: 1 on the diagonal; elsewhere a mix of 0 and 1, 2..n_g, n_g+1..510 (keys >= T lie past the backward's histogram
               plan) and 511 (unreachable);
      walk:    the expected walk (expected_walk(rp) hops of the dominant feature 4), the same with 1, 2 or 3 bytes changed, a fully
               random walk, a walk cut short (zeros before L) or one longer than L; bytes [dk, hops) stay 0."""
    rng = np.random.default_rng(seed)
    rels, pois, edges = [], [], []
    for n in ns:
        C = n * n
        i, j = np.repeat(np.arange(n), n), np.tile(np.arange(n), n)
        cat = rng.choice(4, size=C, p=[0.06, 0.34, 0.34, 0.26])
        key = np.select([cat == 0, cat == 1, cat == 2],
                        [rng.integers(0, 2, C), rng.integers(2, min(max(n, 2), 510) + 1, C), rng.integers(n + 1, 511, C) if n < 510
                         else rng.integers(2, 511, C)], 511)
        key = np.where((cat == 1) & (n < 2), 511, key)
        key = np.where(i == j, 1, key)
        L = expected_walk(key, dk)
        pos = np.arange(hops)[None, :]
        walk = np.where(pos < L[:, None], 4, 0).astype(np.int64)
        mode = rng.choice(7, size=C, p=[0.3, 0.14, 0.1, 0.1, 0.14, 0.11, 0.11])
        feat = _features(rng, (C, hops))
        # 1..3 deviating bytes at distinct positions of [0, dk)
        p0 = rng.integers(0, dk, C)
        steps = [np.zeros(C, np.int64), rng.integers(1, max(dk, 2), C)]
        steps.append((steps[1] + rng.integers(1, max(dk - 1, 2), C)) % max(dk, 1))
        rows = np.arange(C)
        for r in range(3):
            sel = (mode >= r + 1) & (mode <= 3)
            p = (p0 + steps[r]) % dk
            cur = walk[rows, p]
            v = feat[:, r]
            v = np.where(rng.random(C) < 0.15, 0, v)                       # a zero byte: the walk ends early
            v = np.where(v == cur, v % 127 + 1, v)
            walk[rows[sel], p[sel]] = v[sel]
        m4 = mode == 4                                                      # fully random walk, zeros included
        rnd = np.where(rng.random((C, hops)) < 0.1, 0, feat)
        walk[m4] = np.where(pos < dk, rnd, 0)[m4]
        cut = rng.integers(0, np.maximum(L, 1))                             # cut short: zeros from `cut` on
        m5 = (mode == 5)[:, None] & (pos >= cut[:, None]) & (pos < L[:, None])
        walk[m5] = 0
        extra = rng.integers(1, dk + 1, C)                                  # longer than L: bytes [L, L + extra) ∩ [0, dk)
        m6 = (mode == 6)[:, None] & (pos >= L[:, None]) & (pos < (L + extra)[:, None]) & (pos < dk)
        walk[m6] = feat[m6]
        rels.append(key)
        pois.append(rng.integers(0, num_bins, C))
        edges.append(walk)
    n = np.asarray(ns, np.int32)
    sq = np.zeros(len(ns) + 1, np.int64)
    np.cumsum(n.astype(np.int64) ** 2, out=sq[1:])
    h_rel = torch.from_numpy(np.concatenate(rels).astype(np.int16))
    h_poi = torch.from_numpy(np.concatenate(pois).astype(np.int16))
    h_edge = torch.from_numpy(np.concatenate(edges).astype(np.uint8))
    assert int(h_edge.max()) <= 127 and not h_edge[:, dk:].any()
    return SimpleNamespace(B=len(ns), N=int(n.max()), n=torch.from_numpy(n).cuda(), n_host=n, sq_off=torch.from_numpy(sq).cuda(),
                           rel_pos16=h_rel.cuda(), poi_pos16=h_poi.cuda(), edge_in8=h_edge.contiguous().cuda(), hops=hops,
                           dk=dk, rel_pos_max=rel_pos_max, h_rel=h_rel.long(), h_poi=h_poi.long(), h_edge=h_edge.long())


SMALLS = [1, 2, 3, 5, 8, 13, 21, 34, 55, 89, 7, 4]
# (hops, dk, graph sizes, num_bins, rel_pos_max, extra pitch, bf16 layer planes, backward warps planned)
# hops: all eight HOPW instantiations, each with dk = hops and one dk < hops.  T = max n + 1 covers every residue mod 8.
K2_CASES = [
    (4, 4, [1], 64, 1024, 0, 1, 12),                    # T = 2: one node
    (4, 1, [2, 3, 1, 3], 1, 20, 0, 5, 12),              # T = 4
    (8, 8, [12, 5, 1, 9], 1024, 3, 0, 6, 3),            # T = 13
    (8, 3, [13, 2, 7], 64, 1024, 0, 7, 12),             # T = 14
    (12, 12, [14, 14, 3], 1, 1024, 0, 13, 12),          # T = 15
    (12, 5, [15, 8, 1], 1024, 20, 0, 1, 3),             # T = 16
    (16, 16, [16, 4, 11, 16], 64, 3, 0, 5, 12),         # T = 17
    (16, 1, [17, 2], 64, 1024, 24, 6, 12),              # T = 18, pitch 48 > round_up(T, 8)
    (20, 20, [18, 9, 3], 1024, 1024, 0, 7, 3),          # T = 19
    (20, 7, [35, 20, 6], 64, 20, 0, 13, 12),            # T = 36
    (8, 8, [47, 3, 3], 1, 1024, 0, 5, 12),              # T = 48
    (24, 13, [130, 64, 3], 1024, 1024, 0, 5, 2),        # T = 131
    (20, 20, [200, 1, 2], 1, 1024, 0, 6, 9),            # T = 201
    (24, 24, [299, 150, 40, 7], 64, 1024, 0, 1, 6),     # T = 300
    (28, 2, [509, 12], 64, 20, 0, 7, 3),                # T = 510: key 510 is the only one past the plan
    (32, 32, [510, 30], 1, 1024, 0, 13, 4),             # T = 511
    (28, 28, [512] + SMALLS, 1024, 1024, 0, 6, 1),      # T = 513: one 512-node graph and many small ones
    (32, 17, [512] + SMALLS, 64, 3, 0, 1, 3),           # T = 513
]


def _case_id(c):
    return f"h{c[0]}-dk{c[1]}-T{max(c[2]) + 1}-bins{c[3]}-rpm{c[4]}"


def test_case_matrix_covers_every_backward_plan():
    """The cases above run every hop width with dk = hops and dk < hops (dk = 1 included), every T residue mod 8, all three
    rel_pos_max values, and backward warp plans from 1 to 12 — among them the 1-, 2- and 3-warp plans."""
    assert {c[0] for c in K2_CASES} == {4, 8, 12, 16, 20, 24, 28, 32}
    for hops in range(4, 33, 4):
        dks = {c[1] for c in K2_CASES if c[0] == hops}
        assert hops in dks and min(dks) < hops
    assert 1 in {c[1] for c in K2_CASES}
    assert {(max(c[2]) + 1) % 8 for c in K2_CASES} == set(range(8))
    assert {c[4] for c in K2_CASES} == {1024, 20, 3}
    assert {c[3] for c in K2_CASES} == {1, 64, 1024}
    warps = set()
    for hops, dk, ns, bins, rpm, extra, layers, want in K2_CASES:
        got = k2_bwd_plan(max(ns) + 1, hops, bins)[2]
        assert got == want, (hops, ns, bins, got, want)
        warps.add(got)
    assert {1, 2, 3, 4, 6, 12} <= warps, warps


def _bwd_call(pk, dbias, dtype_code, n_layers, layer_stride, T, Tp, E, W, num_bins):
    """mobgt_bias_bwd through the C-ABI (what ops.bias_bwd_raw does, with an explicit plane stride)."""
    from mobgt_b200 import _C
    dev = E.device
    ws_bytes = int(_C.lib().mobgt_bias_bwd_workspace_bytes(T, pk.hops, num_bins))
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


GRAD_NAMES = ("dR", "dPpos", "dE", "dW", "dtvd")


def _check_grads(got, ref, A, tag):
    """|got - ref| <= 2e-5 * A_entry for every entry; dE row 0 (the padding row) is 0 by definition of the kernel."""
    for name, g, r, a in zip(GRAD_NAMES, got, ref, A):
        g = g.detach().double().cpu().reshape(r.shape)
        if name == "dE":
            assert (g[0] == 0).all(), tag
            g, r, a = g[1:], r[1:], a[1:]
        err = (g - r).abs()
        bad = err > 2e-5 * a
        assert not bad.any(), (tag, name, int(bad.sum()), float(err.max()), float((err / a.clamp_min(1e-300)).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("case", K2_CASES, ids=_case_id)
def test_k2_adversarial_fwd_bwd_matches_float64(lib_built, case):
    """mobgt_bias_fwd (fp32 and bf16 output) and mobgt_bias_bwd (one fp32 plane, n_layers bf16 planes, contiguous and strided)
    against k2_reference in float64: forward within 1e-5 * A_cell (bf16: plus 2^-8 |ref|), -inf exactly where rel_pos_max masks;
    every table gradient within 2e-5 * A_entry; dBias cells the kernel must not read set to NaN change no bit of the result."""
    from mobgt_b200 import ops
    hops, dk, ns, bins, rpm, extra, n_layers, want_warps = case
    seed = hops * 1000 + dk * 10 + len(ns)
    pk = adversarial_batch(seed, ns, hops, dk, bins, rpm)
    T = pk.N + 1
    Tp = ops.bias_pitch(T) + extra
    rrows, stride, warps = k2_bwd_plan(T, hops, bins)
    assert warps == want_warps
    # the plan's row layout as the library sizes it: workspace = dEW + (SMs + 1) partial rows + 16 + SMs per-CTA fixed-point
    # tables + the launch-wide fixed-point tables
    ws = int(ops._C.lib().mobgt_bias_bwd_workspace_bytes(T, hops, bins))
    rest = ws - 16 - 4 * hops * 128 * H - 8 * (hops * 128 * H + 512 * H) - 4 * stride
    assert ws > 0 and rest > 0 and rest % (4 * stride + 8 * hops * 16 * H) == 0
    tabs = _tables(bins, hops, seed)
    A_tabs = [x.abs() for x in tabs]
    ref = k2_reference(pk.n_host, pk.h_rel, pk.h_poi, pk.h_edge, dk, rpm, *tabs)
    A = k2_reference(pk.n_host, pk.h_rel, pk.h_poi, pk.h_edge, dk, rpm, *A_tabs)
    live = live_mask(pk.n_host, T).expand_as(ref)
    masked = torch.isneginf(ref) & live
    fin = live & ~masked
    # every walk mode, every key class and both feature ranges occur
    kk = pk.h_rel
    nd = (pk.h_edge != torch.from_numpy(np.where(np.arange(hops)[None, :] < expected_walk(kk.numpy(), dk)[:, None], 4, 0))).sum(1)
    if max(ns) > 1:
        assert (kk == 511).any() and ((kk >= 2) & (kk < 511)).any()
        assert (nd == 0).any() and (nd >= 1).any()
    if sum(k * k - k for k in ns) > 40:
        assert (pk.h_edge >= 16).any() and ((pk.h_edge >= 1) & (pk.h_edge < 16) & (pk.h_edge != 4)).any()
        assert (nd >= min(dk, 3)).any() and (nd == 1).any()
    cu = [x.float().cuda().contiguous() for x in tabs]
    # ---- forward, fp32 and bf16
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
    # ---- backward, fp32 dBias (one summed plane); row 0 and the -inf cells hold values the kernel must not use
    gen = torch.Generator().manual_seed(seed + 1)
    sq = live_mask(pk.n_host, T, Tp).expand(pk.B, H, T, Tp)
    dB = torch.where(sq, torch.randn(pk.B, H, T, Tp, generator=gen), torch.zeros(()))
    used = torch.zeros(pk.B, H, T, Tp, dtype=torch.bool)
    used[..., :T] = fin
    used[:, :, 0, :] = False
    Ecu, Wcu = cu[2], cu[3]
    dB64 = dB[..., :T].double()
    gref = reference_grads(pk, tabs, dB64)
    gA = reference_grads(pk, A_tabs, dB64.abs())
    got32 = ops.bias_bwd_raw(pk, dB.cuda(), Ecu, Wcu, bins)
    _check_grads(got32, gref, gA, "f32")
    # never-read cells: NaN everywhere outside the used cells changes nothing, bit for bit
    dirty = torch.where(used, dB, torch.full((), float("nan")))
    again = ops.bias_bwd_raw(pk, dirty.cuda(), Ecu, Wcu, bins)
    for a_, b_, name in zip(again, got32, GRAD_NAMES):
        assert torch.equal(a_, b_), ("f32 NaN fill", name)
    # ---- backward, n_layers bf16 planes summed inside the kernel; the reference takes the float64 sum of the same values
    planes = torch.stack([(torch.randn(pk.B, H, T, Tp, generator=gen) * (0.5 + 0.25 * l)).to(torch.bfloat16)
                          for l in range(n_layers)])
    planes = torch.where(sq.unsqueeze(0), planes, torch.zeros((), dtype=torch.bfloat16))
    psum = planes.double().sum(0)[..., :T]
    gref16 = reference_grads(pk, tabs, psum)
    gA16 = reference_grads(pk, A_tabs, planes.double().abs().sum(0)[..., :T])
    got16 = ops.bias_bwd_raw(pk, planes.cuda(), Ecu, Wcu, bins)
    _check_grads(got16, gref16, gA16, f"bf16 x{n_layers}")
    nanbf = torch.full((), float("nan"), dtype=torch.bfloat16)
    dirty16 = torch.where(used.unsqueeze(0), planes, nanbf)
    again16 = ops.bias_bwd_raw(pk, dirty16.cuda(), Ecu, Wcu, bins)
    for a_, b_, name in zip(again16, got16, GRAD_NAMES):
        assert torch.equal(a_, b_), ("bf16 NaN fill", name)
    # planes further apart than one plane (layer_stride > B*H*T*Tp), NaN in the gaps: same result bit for bit
    if n_layers in (5, 13):
        plane = pk.B * H * T * Tp
        ls = plane + 40
        flat = torch.full((n_layers * ls,), float("nan"), dtype=torch.bfloat16)
        flat.view(n_layers, ls)[:, :plane] = dirty16.reshape(n_layers, plane)
        flat = flat.cuda()
        gs = _bwd_call(pk, flat, ops.BF16, n_layers, ls, T, Tp, Ecu, Wcu, bins)
        for a_, b_, name in zip(gs, got16, GRAD_NAMES):
            assert torch.equal(a_, b_), ("bf16 strided", name)


@pytest.mark.gpu
def test_k2_backward_bitwise_reproducible_on_rare_path(lib_built):
    """Many deviating bytes, features >= 16 and keys past the plan (the fixed-point atomics of the rare path): three runs,
    fp32 and bf16 planes, give identical bits."""
    from mobgt_b200 import ops
    hops, dk, bins = 24, 24, 64
    pk = adversarial_batch(99, [200, 150, 90, 60, 33, 17, 9], hops, dk, bins, 1024)
    T = pk.N + 1
    Tp = ops.bias_pitch(T)
    tabs = [x.float().cuda().contiguous() for x in _tables(bins, hops, 99)]
    gen = torch.Generator().manual_seed(5)
    sq = live_mask(pk.n_host, T, Tp).expand(pk.B, H, T, Tp)
    dB = torch.where(sq, torch.randn(pk.B, H, T, Tp, generator=gen), torch.zeros(())).cuda()
    planes = torch.where(sq.unsqueeze(0), torch.randn(7, pk.B, H, T, Tp, generator=gen), torch.zeros(())).to(torch.bfloat16).cuda()
    for src in (dB, planes):
        first = ops.bias_bwd_raw(pk, src, tabs[2], tabs[3], bins)
        for _ in range(3):
            again = ops.bias_bwd_raw(pk, src, tabs[2], tabs[3], bins)
            for a_, b_, name in zip(again, first, GRAD_NAMES):
                assert torch.equal(a_, b_), (src.dtype, name)


# ------------------------------------------------------------------------------------- the rel_pos_max mask through K3
def attention64(qkv, bias, tok_off, d=24, drop=None):
    """float64 softmax(q k^T / sqrt(d) + bias) v per packed graph (model_fqandtoyo.py:1693-1706): (out, lse).
    drop = (p, seed): libmobgt's counter-based keep mask (tests/helpers.attn_drop_keep) applied after the softmax."""
    D = H * d
    outs, lses = [], []
    for g in range(len(tok_off) - 1):
        a, e = int(tok_off[g]), int(tok_off[g + 1])
        T = e - a
        q = qkv[a:e, :D].view(T, H, d).transpose(0, 1)
        k = qkv[a:e, D:2 * D].view(T, H, d).transpose(0, 1)
        v = qkv[a:e, 2 * D:].view(T, H, d).transpose(0, 1)
        s = (q * d ** -0.5) @ k.transpose(1, 2) + bias[g, :, :T, :T]
        lses.append(torch.logsumexp(s, -1).t())
        pr = torch.softmax(s, -1)
        if drop is not None:
            masks = [attn_drop_keep(g * H + h, T, drop[0], drop[1]) for h in range(H)]
            keep = torch.from_numpy(np.stack([m[0] for m in masks]))
            pr = pr * keep.to(pr.dtype) * masks[0][1]
        outs.append((pr @ v).transpose(0, 1).reshape(T, D))
    return torch.cat(outs), torch.cat(lses)


def _masked_batch(rel_pos_max):
    """Chains of ~300 distinct POIs (whole 128-column key tiles of a query row fall past rel_pos_max), chains and trajectories of
    at most 15 nodes (the SIMT small-graph kernels), collated at rel_pos_max."""
    from mobgt_b200 import collator, synth
    w = synth.make_world("c1", seed=1)
    items = [_chain_item(w, 300, 1, 0), _chain_item(w, 260, 2, 1), _chain_item(w, 12, 3, 2), _chain_item(w, 15, 4, 3)]
    items += synth.make_items(w, 3, 14, seed=5, start=4) + synth.make_items(w, 2, 80, seed=6, start=7)
    b = collator.collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=rel_pos_max, world=w)
    return w, items, b


def _assert_mask_coverage(bias, tok_off):
    """Some query row of a large graph has an entire 128-column key tile at -inf, and some graph of <= 15 nodes has -inf cells."""
    full_tile = small = False
    for g in range(len(tok_off) - 1):
        Tg = int(tok_off[g + 1] - tok_off[g])
        m = torch.isneginf(bias[g, 0, :Tg, :Tg])
        if Tg <= 16:
            small |= bool(m.any())
        for c0 in range(0, Tg, 128):
            full_tile |= bool(m[:, c0:c0 + 128].all(1).any())
    assert full_tile and small


@pytest.mark.gpu
@pytest.mark.parametrize("rel_pos_max", [20, 3])
@pytest.mark.parametrize("p_drop", [0.0, 0.1])
def test_attention_bf16_on_masked_bias(lib_built, rel_pos_max, p_drop):
    """mobgt_attn_fwd / _bwd (tensor-core and SIMT kernels) on a K2 bias with rel_pos_max -inf cells: out, lse, dqkv finite and
    within the bf16 tolerances of the attention tests against float64; dS exactly 0 on every -inf cell in all three dS modes."""
    from mobgt_b200 import ops
    from test_k2_k3_k4 import tables
    w, items, b = _masked_batch(rel_pos_max)
    R, Pp, E, W, t = tables(seed=13)
    bias = ops.bias_fwd_raw(b, *[x.cuda().contiguous() for x in (R, Pp, E, W.view(-1), t.view(-1))], out_dtype=torch.bfloat16)
    tok_off = b.tok_off.cpu().numpy()
    _assert_mask_coverage(bias.cpu(), tok_off)
    ntok = int(b.tok_pos.numel())
    gen = torch.Generator().manual_seed(41)
    qkv = (torch.randn(ntok, 3 * 192, generator=gen) * 1.2).to(torch.bfloat16)
    dout = torch.randn(ntok, 192, generator=gen).to(torch.bfloat16)
    seed = 0x5DEECE66D if p_drop > 0 else 0
    out, lse = ops.attn_fwd_raw(qkv.cuda(), bias, b, drop_p=p_drop, seed=seed)
    db0 = torch.full(bias.shape, float("nan"), dtype=torch.float32, device="cuda")
    dq0 = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, db0, 0, drop_p=p_drop, seed=seed)
    db1 = db0.clone()
    dq1 = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, db1, 1, drop_p=p_drop, seed=seed)
    plane = torch.full(bias.shape, float("nan"), dtype=torch.bfloat16, device="cuda")
    dq2 = ops.attn_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, plane, 2, drop_p=p_drop, seed=seed)
    torch.cuda.synchronize()
    for x in (out, lse, dq0):
        assert torch.isfinite(x).all()
    assert torch.equal(dq0, dq2)
    q64 = qkv.double().requires_grad_(True)
    b64 = bias.double().cpu().requires_grad_(True)
    ref, ref_lse = attention64(q64, b64, tok_off, drop=(p_drop, seed) if p_drop > 0 else None)
    (ref * dout.double()).sum().backward()
    assert (out.double().cpu() - ref.detach()).abs().max().item() <= 2e-2 * max(1.0, ref.abs().max().item())
    assert (lse.double().cpu() - ref_lse.detach()).abs().max().item() <= 2e-2
    gq = q64.grad
    assert (dq0.double().cpu() - gq).abs().max().item() <= 2e-2 * max(1.0, gq.abs().max().item())
    biasc, db0c, db1c, planec = bias.cpu(), db0.cpu(), db1.cpu(), plane.cpu()
    for g in range(b.B):
        Tg = int(tok_off[g + 1] - tok_off[g])
        m = torch.isneginf(biasc[g, :, :Tg, :Tg])
        got = db0c[g, :, :Tg, :Tg]
        gb = b64.grad[g, :, :Tg, :Tg]
        assert torch.isfinite(got).all(), g
        assert (got[m] == 0).all() and (planec[g, :, :Tg, :Tg][m] == 0).all(), g
        assert (got.double() - gb).abs().max().item() <= 2e-2 * max(1.0, gb.abs().max().item()), g
        got1 = db1c[g, :, :Tg, :Tg]                                             # mode 1 adds onto mode 0's values
        assert torch.allclose(got1, 2 * got, rtol=1e-6, atol=1e-7) and (got1[m] == 0).all(), g
        assert torch.equal(planec[g, :, :Tg, :Tg].float(), got.to(torch.bfloat16).float()), g


@pytest.mark.gpu
@pytest.mark.parametrize("rel_pos_max", [20, 3])
@pytest.mark.parametrize("p_drop", [0.0, 0.1])
def test_attention_f32_on_masked_bias(lib_built, rel_pos_max, p_drop):
    """mobgt_attn_f32_fwd / _bwd on an fp32 K2 bias with rel_pos_max -inf cells: within 1e-5 of float64, dS exactly 0 on -inf."""
    from mobgt_b200 import ops
    from test_k2_k3_k4 import tables
    w, items, b = _masked_batch(rel_pos_max)
    R, Pp, E, W, t = tables(seed=14)
    bias = ops.bias_fwd_raw(b, *[x.cuda().contiguous() for x in (R, Pp, E, W.view(-1), t.view(-1))], out_dtype=torch.float32)
    tok_off = b.tok_off.cpu().numpy()
    _assert_mask_coverage(bias.cpu(), tok_off)
    ntok = int(b.tok_pos.numel())
    gen = torch.Generator().manual_seed(43)
    qkv = torch.randn(ntok, 3 * 192, generator=gen) * 1.2
    dout = torch.randn(ntok, 192, generator=gen)
    seed = 0x0123456789ABCDEF if p_drop > 0 else 0
    out, lse = ops.attn_f32_fwd_raw(qkv.cuda(), bias, b, drop_p=p_drop, seed=seed)
    db = torch.full(bias.shape, 7.0, dtype=torch.float32, device="cuda")
    dq = ops.attn_f32_bwd_raw(qkv.cuda(), bias, out, dout.cuda(), lse, b, db, 0, drop_p=p_drop, seed=seed)
    torch.cuda.synchronize()
    for x in (out, lse, dq):
        assert torch.isfinite(x).all()
    q64 = qkv.double().requires_grad_(True)
    b64 = bias.double().cpu().requires_grad_(True)
    ref, ref_lse = attention64(q64, b64, tok_off, drop=(p_drop, seed) if p_drop > 0 else None)
    (ref * dout.double()).sum().backward()
    tol = 1e-5
    assert (out.double().cpu() - ref.detach()).abs().max().item() <= tol * max(1.0, ref.abs().max().item())
    assert (lse.double().cpu() - ref_lse.detach()).abs().max().item() <= tol * max(1.0, ref_lse.abs().max().item())
    gq = q64.grad
    assert (dq.double().cpu() - gq).abs().max().item() <= tol * max(1.0, gq.abs().max().item())
    biasc, dbc = bias.cpu(), db.cpu()
    for g in range(b.B):
        Tg = int(tok_off[g + 1] - tok_off[g])
        m = torch.isneginf(biasc[g, :, :Tg, :Tg])
        got = dbc[g, :, :Tg, :Tg]
        gb = b64.grad[g, :, :Tg, :Tg]
        assert torch.isfinite(got).all() and (got[m] == 0).all(), g
        assert (got.double() - gb).abs().max().item() <= tol * max(1.0, gb.abs().max().item()), g


# --------------------------------------------------------------------------------------- the rel_pos_max mask, model level
def _pair_masked(precision, rel_pos_max=20):
    """oracle and product Graphormer with the same weights, items collated at rel_pos_max on both sides (cf. test_round2_gpu._pair)."""
    from mobgt_b200 import collator, model, synth
    dataset_name = "gowalla_nevda"
    w = synth.make_world("c1", seed=1, dataset_name=dataset_name)
    items = synth.make_items(w, 6, 40, seed=12) + [_chain_item(w, 45, 21, 6), _chain_item(w, 26, 22, 7), _chain_item(w, 9, 23, 8)]
    hp = dict(n_layers=2, num_heads=8, hidden_dim=128, dropout_rate=0.0, intput_dropout_rate=0.0, weight_decay=0.01, ffn_dim=256,
              warmup_updates=10, tot_updates=100, peak_lr=2e-4, end_lr=1e-9, edge_type="multi_hop", multi_hop_max_dist=20,
              attention_dropout_rate=0.0)
    torch.manual_seed(3)
    om = mo.Graphormer(w, n_layers=2, ffn_dim=256, dataset_name=dataset_name, multi_hop_max_dist=20).eval()
    with torch.no_grad():
        for emb in (om.edge_encoder, om.rel_pos_encoder, om.poi_pos_encoder):
            emb.weight.mul_(0.3)
            emb.weight[0].zero_()
        om.edge_dis_encoder.weight.mul_(0.3)
    pm = model.Graphormer(dataset_name=dataset_name, world=w, precision=precision, **hp).cuda().eval()
    missing, _ = pm.load_state_dict(om.state_dict(), strict=False)
    assert not missing, missing
    ob = mo.collate([mo.preprocess_item(it, hop_cap=20) for it in items], w, multi_hop_max_dist=20, rel_pos_max=rel_pos_max)
    pb = collator.collator_toyota(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=rel_pos_max, world=w)
    return w, items, om, pm, ob, pb


@pytest.mark.gpu
def test_collated_attn_bias_view_at_rel_pos_max_20(lib_built):
    """The packed batch's reference-shaped attn_bias view (collator.py:354-358 mask included) == the oracle collator's."""
    w, items, om, pm, ob, pb = _pair_masked(16)
    got = pb.attn_bias.cpu()
    assert got.shape == ob.attn_bias.shape and torch.equal(got, ob.attn_bias)
    n = pb.n_host
    inner = torch.stack([torch.isneginf(ob.attn_bias[g, 1:int(n[g]) + 1, 1:int(n[g]) + 1]).any() for g in range(len(n))])
    assert inner[-3:].all()                 # the chains (the last three items) have masked pairs
    assert torch.equal(pb.rel_pos.cpu(), ob.rel_pos)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [16, 32])
def test_model_at_rel_pos_max_20_matches_oracle(lib_built, precision):
    """Graphormer at rel_pos_max = 20 (the default of the reference's collators) against the oracle: logits, loss and every
    parameter gradient.  precision 16: logits and loss within 2e-2, gradients as in test_model_parity (5e-2 norm-wise, no
    element off by more than 12 % of the tensor's largest entry, through two bf16 encoder layers).  precision 32: logits and
    loss within 1e-5; gradients within 1e-5 of the fp32 oracle or of its float64 run (test_fp32_mode), or, where masking makes
    a gradient so ill-conditioned that the fp32 oracle itself is far from float64, within 2.5 x that distance (see below)."""
    from test_fp32_mode import _oracle_float64
    w, items, om, pm, ob, pb = _pair_masked(precision)
    tol = 2e-2 if precision == 16 else 1e-5
    try:
        with torch.no_grad():
            ref = om(ob)
            got = pm(pb)
        for a, r in zip(got, ref):
            assert a.shape == r.shape and torch.isfinite(a).all()
            assert (a.float().cpu() - r).abs().max().item() <= tol * max(1.0, r.abs().max().item())
        for m_ in (om, pm):
            m_.train()
            m_.poi_distance_model.eval()
            m_.poi_cat_model.eval()
        pm.pos_embed.p = 0.0
        lref = om.training_loss(ob)
        lref.backward()
        lgot = pm.training_step(pb)
        lgot.backward()
        assert abs(lgot.item() - lref.item()) <= tol * abs(lref.item()), (lgot.item(), lref.item())
        ref_g = {k: p.grad for k, p in om.named_parameters() if p.grad is not None}
        got_g = {k: p.grad.float().cpu() for k, p in pm.named_parameters() if p.grad is not None}
        ref64 = _oracle_float64(om, ob)[1] if precision == 32 else None
        table = {}
        gmax = max(r.abs().max().item() for r in ref_g.values())
        bad, checked = [], 0
        for k, r in ref_g.items():
            g = got_g.get(k)
            if g is None:
                assert r.abs().max().item() == 0.0, k
                continue
            assert torch.isfinite(g).all(), k
            scale = r.abs().max().item()
            if scale < 1e-6 * gmax:       # mathematically-zero gradients (softmax ignores a per-row constant): rounding noise only
                assert g.abs().max().item() < 1e-3 * gmax, k
                continue
            checked += 1
            normwise = (g - r).norm().item() / r.norm().item()
            if precision == 16:
                elem = (g - r).abs().max().item() / scale
                if normwise > 5e-2 or elem > 0.12:
                    bad.append((k, normwise, elem))
            else:
                # ours against the fp32 oracle and against its float64 run, and the fp32 oracle's own rounding.  With most pairs
                # masked, the edge-table gradients are sums of dS that nearly cancel (every row of dS sums to zero), so fp32
                # rounding of any implementation comes close to 1e-5 there.  Measured on a B200: edge_encoder.weight is 1.19e-5
                # from the fp32 oracle and 1.05e-5 from float64, while the fp32 oracle itself is 4.25e-6 from float64 (other
                # tables: ~7e-7).  So a gradient also passes when it is no further from float64 than 2.5 x the fp32 oracle is
                # (the factor test_round2_gpu.test_canonical_model_on_baseline_shapes allows against the oracle's own error).
                r64 = ref64[k]
                e64 = (g.double() - r64).norm().item() / r64.norm().item()
                o64 = (r.double() - r64).norm().item() / r64.norm().item()
                table[k] = (normwise, e64, o64)
                if min(normwise, e64) > max(tol, 2.5 * o64):
                    bad.append((k, normwise, e64, o64))
        assert checked > 40
        if precision == 32:
            worst = sorted(table, key=lambda k: -table[k][1])[:5]
            print("fp32 gradient errors (ours vs fp32 oracle, ours vs float64 oracle, fp32 oracle vs float64 oracle):",
                  {k: ["%.2e" % v for v in table[k]] for k in worst})
        assert not bad, bad
    finally:
        if precision == 32:
            from mobgt_b200 import ops
            ops.enable_tf32(True)        # leave the process-wide cuBLAS switch as the bf16-mode tests expect it
