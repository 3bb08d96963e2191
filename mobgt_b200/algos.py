"""Drop-in for the reference's Cython module `algos` (/root/reference/graphormer/algos.pyx),
running on the B200 through libmobgt (csrc/k1_apsp.cu).

    floyd_warshall(adjacency_matrix)            algos.pyx:9-54
    gen_edge_input(max_dist, path, edge_feat)   algos.pyx:65-96

plus the batched, device-resident form the rest of this package uses
(`apsp_edge_input_packed`).  Same names, argument meaning and assertion behaviour as the
reference; results are bit-exact (tests/test_k1_apsp.py).  No CPU fallback.
"""
import numpy as np
import torch

from . import _C

UNREACHABLE = 510
# size classes: one launch per class so that tiny graphs do not inherit the block / cluster
# shape of the largest one.  (512, 1024] is the plan for graphs the model cannot take (K1 only: the
# algos drop-in); its walk reads `path`, so that class always gets a path buffer.
_CLASSES = (8, 16, 32, 64, 128, 184, 256, 512, _C.MAX_APSP_NODES)


def pack_graphs(n_host):
    """n[G] -> (n i32, sq_off i64 [G+1], node_off i64 [G+1]) as numpy."""
    n = np.asarray(n_host, np.int32)
    sq = np.zeros(len(n) + 1, np.int64)
    np.cumsum(n.astype(np.int64) ** 2, out=sq[1:])
    no = np.zeros(len(n) + 1, np.int64)
    np.cumsum(n.astype(np.int64), out=no[1:])
    return n, sq, no


def hop_stride(multi_hop_max_dist):
    """Bytes per packed edge_in row for a given multi_hop_max_dist (1..32): the next multiple of 4 (the kernels move walk
    bytes as 32-bit words); the slots past multi_hop_max_dist are never walked and stay "no hop"."""
    dk = int(multi_hop_max_dist)
    if not 1 <= dk <= 32:
        raise ValueError(f"multi_hop_max_dist={dk}: libmobgt supports 1..32 hop slots")
    return (dk + 3) // 4 * 4


def apsp_edge_input_packed(feat, n_dev, sq_off_dev, n_host, hops, shift=0, want_path=False, want_edges=True, dk=None):
    """Batched K1 on device-resident packed graphs.

    feat u8 [sum n^2] (0 = no edge) ; n_dev i32 [G] ; sq_off_dev i64 [G(+1)] ; n_host: numpy copy of n
    hops: bytes per edge_in row (multiple of 4); dk: hop slots walked (multi_hop_max_dist, default = hops).
    Returns dict(dist i16, path i16|None, edge_in u8 [sum n^2, hops]|None, maxdist i32 [G])."""
    dk = int(hops if dk is None else dk)
    _C.require_cuda()
    dev = feat.device
    G = int(n_dev.numel())
    cells = int(feat.numel())
    dist = torch.empty(cells, dtype=torch.int16, device=dev)
    path = torch.empty(cells, dtype=torch.int16, device=dev) if want_path else None
    edge_in = torch.empty((cells, hops), dtype=torch.uint8, device=dev) if want_edges else None
    maxdist = torch.zeros(G, dtype=torch.int32, device=dev)
    n_host = np.asarray(n_host)
    if G == 0:
        return dict(dist=dist, path=path, edge_in=edge_in, maxdist=maxdist)
    if (n_host < 1).any() or (n_host > _CLASSES[-1]).any():
        raise ValueError(f"node counts must be in [1, {_CLASSES[-1]}]")
    lo = 0
    s = _C.stream_ptr()
    for hi in _CLASSES:
        sel = np.nonzero((n_host > lo) & (n_host <= hi))[0]
        lo = hi
        if len(sel) == 0:
            continue
        if len(sel) == G:
            gids = None
        else:
            gids = torch.from_numpy(sel.astype(np.int32)).to(dev, non_blocking=True)
        p = path
        if p is None and hi > _C.MAX_NODES:
            p = torch.empty(cells, dtype=torch.int16, device=dev)     # the walk's input; freed after the call (stream-ordered)
        _C.call("mobgt_apsp_edge_input", _C.ptr(feat), _C.ptr(n_dev), _C.ptr(sq_off_dev), _C.ptr(gids),
                int(len(sel)), int(n_host[sel].max()), int(hops), dk, int(shift),
                _C.ptr(dist), _C.ptr(p), _C.ptr(edge_in), _C.ptr(maxdist), s)
    return dict(dist=dist, path=path, edge_in=edge_in, maxdist=maxdist)


def floyd_warshall(adjacency_matrix):
    """algos.pyx:9-54.  [n,n] bool/int array -> (M int64 [n,n], path int64 [n,n]), 510 = unreachable."""
    a = np.asarray(adjacency_matrix)
    (nrows, ncols) = a.shape
    assert nrows == ncols
    n = nrows
    if n == 0:
        return np.zeros((0, 0), np.int64), np.zeros((0, 0), np.int64)
    feat = torch.from_numpy(np.ascontiguousarray(a != 0, dtype=np.uint8).reshape(-1)).cuda()
    nn, sq, _ = pack_graphs([n])
    out = apsp_edge_input_packed(feat, torch.from_numpy(nn).cuda(), torch.from_numpy(sq).cuda(), nn,
                                 hops=4, shift=0, want_path=True, want_edges=False)
    M = out["dist"].cpu().numpy().astype(np.int64).reshape(n, n)
    path = out["path"].cpu().numpy().astype(np.int64).reshape(n, n)
    return M, path


def gen_edge_input(max_dist, path, edge_feat):
    """algos.pyx:65-96.  -> float32 [n, n, max_dist, F], -1 where the walk has no hop."""
    path = np.asarray(path)
    edge_feat = np.asarray(edge_feat)
    (nrows, ncols) = path.shape
    assert nrows == ncols
    n = nrows
    max_dist = int(max_dist)
    F = edge_feat.shape[-1]
    if F != 1:
        raise NotImplementedError("libmobgt supports one edge feature per edge (every MobGT dataset has F == 1)")
    if edge_feat.size and (edge_feat.min() < 0 or edge_feat.max() > 254):
        raise ValueError("edge features must lie in [0, 254]")
    if n == 0 or max_dist == 0:
        return -1 * np.ones([n, n, max_dist, F], dtype=np.float32)
    _C.require_cuda()
    p16 = torch.from_numpy(np.ascontiguousarray(path, dtype=np.int16).reshape(-1)).cuda()
    f8 = torch.from_numpy(np.ascontiguousarray(edge_feat[..., 0], dtype=np.uint8).reshape(-1)).cuda()
    nn, sq, _ = pack_graphs([n])
    e = torch.empty((n * n, max_dist), dtype=torch.uint8, device="cuda")
    n_dev, sq_dev = torch.from_numpy(nn).cuda(), torch.from_numpy(sq).cuda()   # keep alive across the call
    _C.call("mobgt_gen_edge_input", _C.ptr(p16), _C.ptr(f8), _C.ptr(n_dev), _C.ptr(sq_dev), 1, n, max_dist, 0,
            _C.ptr(e), _C.stream_ptr())
    raw = e.cpu().numpy()
    out = raw.astype(np.float32)
    out[raw == 255] = -1.0          # 255 == (uint8)(-1): "no hop"
    return out.reshape(n, n, max_dist, 1)
