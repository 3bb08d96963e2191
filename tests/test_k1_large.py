"""K1 on graphs of 513..1024 nodes (csrc/k1_apsp.cu: k1_apsp_large_kernel + k1_walk_from_path_kernel): the algos drop-in takes
every graph the reference's algos.pyx takes on its own data set.

Bit-exact means equal to the C oracle (oracle/algos_oracle.c) in M, path and edge_input, driven like wrapper.py:55-60 via
helpers.run_algos.  The ABI tests run on the CPU (bad arguments are refused before any device work)."""
import ctypes
import os

import numpy as np
import pytest
import torch

import algos_oracle
from helpers import dense_inputs, run_algos

HOPS = 20
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def pack(graphs):
    """graphs: list of (n, src, dst, cnt) -> feat u8 packed, n, sq_off (numpy)."""
    from mobgt_b200.algos import pack_graphs
    n, sq, _ = pack_graphs([g[0] for g in graphs])
    feat = np.zeros(int(sq[-1]), np.uint8)
    for gi, (nn, s, d, c) in enumerate(graphs):
        feat[sq[gi]:sq[gi + 1]].reshape(nn, nn)[s, d] = c + 2
    return feat, n, sq


def run_gpu(graphs, shift=0, want_path=True, hops=HOPS, dk=None):
    from mobgt_b200.algos import apsp_edge_input_packed
    feat, n, sq = pack(graphs)
    out = apsp_edge_input_packed(torch.from_numpy(feat).cuda(), torch.from_numpy(n).cuda(), torch.from_numpy(sq).cuda(), n,
                                 hops=hops, shift=shift, want_path=want_path, dk=dk)
    torch.cuda.synchronize()
    return {k: (v.cpu().numpy() if v is not None else None) for k, v in out.items()}, n, sq


def cells(res, key, n, sq, gi):
    nn, a, b = int(n[gi]), int(sq[gi]), int(sq[gi + 1])
    return res[key][a:b].reshape(nn, nn, *res[key].shape[1:])


def expect_edges(e20, hops, dk, shift):
    """The oracle's first HOPS hop slots (int8, -1 = no hop) as K1 stores them: u8 [n, n, hops], slots >= dk "no hop", + shift."""
    out = np.full(e20.shape[:2] + (hops,), (shift - 1) & 0xFF, np.uint8)
    out[:, :, :dk] = ((e20[:, :, :dk].astype(np.int16) + shift) & 0xFF).astype(np.uint8)
    return out


def check_vs_oracle(res, n, sq, gi, ref, want_path=True, hops=HOPS, dk=HOPS, shift=0):
    Mo, Po, eo, md = ref
    nn = int(n[gi])
    assert (cells(res, "dist", n, sq, gi) == Mo + shift).all(), f"dist differs, graph {gi} n={nn}"
    if want_path:
        assert (cells(res, "path", n, sq, gi) == Po).all(), f"path differs, graph {gi} n={nn}"
    assert (cells(res, "edge_in", n, sq, gi) == expect_edges(eo, hops, dk, shift)).all(), f"edge_input differs, graph {gi} n={nn}"
    assert int(res["maxdist"][gi]) == md


def hub_graph(n, hub, seed, dens=0.003, p_hub=0.3):
    rng = np.random.default_rng(seed)
    a = rng.random((n, n)) < dens
    a[hub, rng.random(n) < p_hub] = True
    a[rng.random(n) < p_hub, hub] = True
    s, d = np.nonzero(a)
    return (n, s, d, rng.integers(1, 100, size=len(s)))


# ---- ABI (CPU) ---------------------------------------------------------------------------------------------------------------
def _buf():
    return ctypes.create_string_buffer(64)     # never dereferenced: the arguments are refused before any device work


def test_n_max_above_1024_is_refused(lib_built):
    from mobgt_b200 import _C
    L = _C.lib()
    b = [_buf() for _ in range(8)]
    p = [ctypes.addressof(x) for x in b]
    rc = L.mobgt_apsp_edge_input(p[0], p[1], p[2], None, 1, 1025, 20, 20, 0, p[3], p[4], p[5], p[6], None)
    assert rc == -1 and "1024" in _C.last_error()                                       # MOBGT_ERR_BAD_SHAPE
    rc = L.mobgt_gen_edge_input(p[0], p[1], p[2], p[3], 1, 1025, 20, 0, p[4], None)
    assert rc == -1 and "1024" in _C.last_error()


def test_large_plan_needs_a_path_buffer(lib_built):
    from mobgt_b200 import _C
    L = _C.lib()
    b = [_buf() for _ in range(8)]
    p = [ctypes.addressof(x) for x in b]
    rc = L.mobgt_apsp_edge_input(p[0], p[1], p[2], None, 1, 600, 20, 20, 0, p[3], None, p[5], p[6], None)
    assert rc == -6 and "path" in _C.last_error()                                       # MOBGT_ERR_NULL


def test_header_limits_match_binding():
    from mobgt_b200 import _C
    src = open(os.path.join(ROOT, "include", "mobgt.h")).read()
    assert f"#define MOBGT_MAX_APSP_NODES {_C.MAX_APSP_NODES} " in src
    assert f"#define MOBGT_MAX_NODES {_C.MAX_NODES} " in src


@pytest.mark.gpu
def test_packed_refuses_1025_nodes(lib_built):
    from mobgt_b200.algos import apsp_edge_input_packed
    n = np.array([1025], np.int32)
    f = torch.zeros(1025 * 1025, dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="1024"):
        apsp_edge_input_packed(f, torch.from_numpy(n).cuda(), torch.tensor([0, 1025 * 1025], device="cuda"), n, hops=20)


@pytest.mark.gpu
def test_model_collation_keeps_the_512_cap(lib_built):
    """K1 takes 1024 nodes, but the collator feeds K2 / K3, which take 512: a larger graph is still refused there."""
    from mobgt_b200 import collator, owndata
    world, splits = owndata.unpack_dataset(np.load(os.path.join(ROOT, "tests", "golden", "gowalla_nevda_real.npz")))
    items = [splits["train"][1559]]                         # 626 nodes
    with pytest.raises(ValueError, match="512"):
        collator.collator_gowalla(items, max_node=1024, multi_hop_max_dist=20, rel_pos_max=1024, world=world)


# ---- bit-exact against the oracle (GPU) --------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_chain_1024_sentinel(lib_built):
    """Directed chain of 1024 nodes: true distances >= 510 read as unreachable, as at 512."""
    n = 1024
    g = (n, np.arange(n - 1), np.arange(1, n), np.ones(n - 1, np.int64))
    res, nn, sq = run_gpu([g])
    M, P = cells(res, "dist", nn, sq, 0), cells(res, "path", nn, sq, 0)
    assert M[0, 509] == 509 and M[0, 510] == 510 and M[500, 1009] == 509 and M[500, 1010] == 510 and M[1023, 0] == 510
    assert P[0, 509] == 508 and P[0, 510] == 510
    check_vs_oracle(res, nn, sq, 0, run_algos(algos_oracle, *g, hop_cap=HOPS))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [513, 777, 1024])
def test_node_510_hub(lib_built, n):
    """Pairs whose last improving intermediate is node 510 carry path == 510 and are skipped by gen_edge_input
    (algos.pyx:87-88), while walks of other pairs still pass through node 510."""
    g = hub_graph(n, 510, seed=1510 + n)
    ref = run_algos(algos_oracle, *g, hop_cap=HOPS)
    Mo, Po = ref[0], ref[1]
    assert ((Po == 510) & (Mo < 510)).sum() > 100, "fixture must exercise the path == 510 collision"
    res, nn, sq = run_gpu([g, g])           # twice: the second copy runs as another cluster of the same launch
    for gi in range(2):
        check_vs_oracle(res, nn, sq, gi, ref)


@pytest.mark.gpu
def test_node_0_hub(lib_built):
    """Improvements through k = 0 leave path == 0, which the reference reads as "direct" (algos.pyx:59-60)."""
    g = hub_graph(700, 0, seed=700)
    ref = run_algos(algos_oracle, *g, hop_cap=HOPS)
    Mo, Po = ref[0], ref[1]
    assert ((Po == 0) & (Mo > 1) & (Mo < 510)).sum() > 100, "fixture must route pairs through node 0"
    res, nn, sq = run_gpu([g])
    check_vs_oracle(res, nn, sq, 0, ref)


@pytest.fixture(scope="module")
def mixed():
    """Large graphs at three densities, mixed with small graphs of every size class, and their oracle results."""
    rng = np.random.default_rng(1024)
    graphs = []
    sizes = [(513, 0.004), (int(rng.integers(514, 1024)), 0.0015), (int(rng.integers(514, 1024)), 0.006), (1024, 0.02),
             (int(rng.integers(514, 1024)), 0.004)]
    small = [1, 2, 7, 12, 30, 60, 100, 150, 200, 300, 511, 512]
    for k, n in enumerate(small):
        graphs.append((n, 0.05 if n < 100 else 0.006))
        if k % 3 == 2 and sizes:
            graphs.append(sizes.pop(0))
    graphs += sizes
    out = []
    for n, dens in graphs:
        a = rng.random((n, n)) < dens
        s, d = np.nonzero(a)
        out.append((n, s, d, rng.integers(1, 100, size=len(s))))
    assert sum(g[0] > 512 for g in out) == 5
    return out, [run_algos(algos_oracle, *g, hop_cap=HOPS) for g in out]


@pytest.mark.gpu
@pytest.mark.parametrize("want_path", [False, True])
@pytest.mark.parametrize("shift", [0, 1])
@pytest.mark.parametrize("hops,dk", [(20, 20), (8, 5)])
def test_mixed_sizes_vs_oracle(lib_built, mixed, want_path, shift, hops, dk):
    """One apsp_edge_input_packed call over every size class (gids select each class's graphs)."""
    graphs, refs = mixed
    res, n, sq = run_gpu(graphs, shift=shift, want_path=want_path, hops=hops, dk=dk)
    assert (res["path"] is None) == (not want_path)
    for gi in range(len(graphs)):
        check_vs_oracle(res, n, sq, gi, refs[gi], want_path=want_path, hops=hops, dk=dk, shift=shift)


@pytest.mark.gpu
def test_mixed_sizes_deterministic(lib_built, mixed):
    graphs, _ = mixed
    a, _, _ = run_gpu(graphs, shift=1, want_path=True)
    b, _, _ = run_gpu(graphs, shift=1, want_path=True)
    for k in ("dist", "path", "edge_in", "maxdist"):
        assert a[k].tobytes() == b[k].tobytes(), k


@pytest.mark.gpu
@pytest.mark.parametrize("traj,n,md,p510", [(1559, 626, 510, 27), (1589, 814, 85, 1)])
def test_real_gowalla_trajectories_dropin(lib_built, traj, n, md, p510):
    """The two train trajectories of the shipped Gowalla-Nevada data set above 512 nodes, through the per-item drop-in exactly
    as wrapper.py:55-60 calls it: floyd_warshall, then gen_edge_input at the full max_dist (510 and 85 hop slots)."""
    from mobgt_b200 import algos, owndata
    z = np.load(os.path.join(ROOT, "tests", "golden", "gowalla_nevda_real.npz"))
    _, splits = owndata.unpack_dataset(z)
    it = splits["train"][traj]
    assert len(it.x) == n
    ei = np.asarray(it.edge_index)
    adj, ef = dense_inputs(n, ei[0], ei[1], np.asarray(it.edge_attr).reshape(-1))
    M, path = algos.floyd_warshall(adj)
    Mo, po = algos_oracle.floyd_warshall(adj)
    assert M.dtype == np.int64 and path.dtype == np.int64
    assert (M == Mo).all() and (path == po).all()
    assert int(M.max()) == md and int(((path == 510) & (M < 510)).sum()) == p510
    e = algos.gen_edge_input(md, path, ef)
    eo = algos_oracle.gen_edge_input(md, po, ef)
    assert e.dtype == np.float32 and e.shape == eo.shape == (n, n, md, 1)
    assert np.array_equal(e, eo)
