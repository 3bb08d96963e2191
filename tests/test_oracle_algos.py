"""CPU: pin the oracle (oracle/algos_oracle.c) to the reference's own outputs.

The golden fixture (tests/golden/algos_golden.npz) was produced by the unmodified, Cython-compiled
/root/reference/graphormer/algos.pyx (tests/golden/make_golden.py).  The reference ships no tests of
its own (SURVEY.md §4), so these vectors are the pin."""
import numpy as np

import algos_oracle
from helpers import digest, golden_graph, run_algos

UNREACH = 510


class RestatedAlgos:
    """algos.pyx:9-96 (SURVEY.md A1a-A1c) restated in numpy / Python, independently of oracle/algos_oracle.c: the stand-in for
    the compiled reference where oracle/_ref is not built.  test_restatement_matches_the_reference_golden pins it to the
    outputs the compiled reference produced (tests/golden/algos_golden.npz)."""

    @staticmethod
    def floyd_warshall(adjacency_matrix):
        M = np.array(adjacency_matrix, dtype=np.int64)
        n = M.shape[0]
        path = np.zeros((n, n), np.int64)
        M[M == 0] = UNREACH                                  # :27-32: zero entries -> 510, the diagonal -> 0
        np.fill_diagonal(M, 0)
        for k in range(n):                                   # :35-45: k ascending, strict '>', path = the last improving k
            cand = M[:, k:k + 1] + M[k:k + 1, :]             # (row and column k cannot change while k is the intermediate)
            better = M > cand
            M[better] = cand[better]
            path[better] = k
        unreach = M >= UNREACH                               # :48-52
        M[unreach] = UNREACH
        path[unreach] = UNREACH
        return M, path

    @staticmethod
    def get_all_edges(path, i, j):
        k = int(path[i, j])                                  # :57-62: in-order expansion; k == 0 stops (the node-0 quirk)
        if k == 0:
            return []
        return RestatedAlgos.get_all_edges(path, i, k) + [k] + RestatedAlgos.get_all_edges(path, k, j)

    @staticmethod
    def gen_edge_input(max_dist, path, edge_feat, hop_cap=None):
        """:65-96; hop_cap = the reference's output sliced [:, :, :hop_cap] (collator.py:323)."""
        path = np.asarray(path, dtype=np.int64)
        edge_feat = np.asarray(edge_feat, dtype=np.int64)
        n, F = path.shape[0], edge_feat.shape[-1]
        hops = int(max_dist) if hop_cap is None else min(int(max_dist), int(hop_cap))
        out = np.full((n, n, hops, F), -1, np.float32)
        for i in range(n):
            for j in range(n):
                if i == j or path[i, j] == UNREACH:          # only the top-level entry is compared with 510
                    continue
                walk = [i] + RestatedAlgos.get_all_edges(path, i, j) + [j]
                for h in range(min(len(walk) - 1, hops)):
                    out[i, j, h] = edge_feat[walk[h], walk[h + 1]]
        return out


def _reference():
    """The compiled reference (oracle/_ref) when it was built, else the restatement pinned to its golden outputs."""
    import build_ref
    ref = build_ref.load()
    return RestatedAlgos if ref is None else ref


def test_kats_full_arrays(golden):
    names = [str(x) for x in golden["names"]]
    checked = 0
    for key in golden.files:
        if not key.endswith("_M") or not key.startswith("full_"):
            continue
        name = key[len("full_"):-2]
        idx = names.index(name)
        _, n, s, d, c = golden_graph(golden, idx)
        M, path, e20, md = run_algos(algos_oracle, n, s, d, c, hop_cap=20)
        assert (M == golden[f"full_{name}_M"]).all(), name
        assert (path == golden[f"full_{name}_path"]).all(), name
        assert (e20 == golden[f"full_{name}_e20"]).all(), name
        assert md == int(golden["max_dist"][idx])
        checked += 1
    assert checked >= 30


def test_survey_kats_by_value(golden):
    """SURVEY.md §8c KAT-A / KAT-B / KAT-C literal values."""
    a = golden["full_kat_a_M"]
    assert a.tolist() == [[0, 1, 2, 3, 4], [510, 0, 1, 2, 3], [510, 2, 0, 1, 2], [510, 1, 2, 0, 1], [510, 510, 510, 510, 0]]
    assert golden["full_kat_a_path"].tolist() == [[0, 0, 1, 2, 3], [510, 0, 0, 2, 3], [510, 3, 0, 0, 3], [510, 0, 1, 0, 0],
                                                  [510, 510, 510, 510, 0]]
    assert golden["full_kat_a_e20"][0, 3, :5].tolist() == [3, 3, 3, -1, -1]
    assert golden["full_kat_b_node0_e20"][1, 2, :3].tolist() == [0, -1, -1]      # node-0 quirk
    assert golden["full_kat_c_cycle_e20"][2, 1, :2].tolist() == [0, -1]


def test_all_digests(golden):
    """Every fixture graph (hand KATs, random digraphs, all 4 959 real Gowalla-Nevada train graphs n<=256)."""
    G = len(golden["n"])
    bad = []
    for idx in range(G):
        _, n, s, d, c = golden_graph(golden, idx)
        M, path, e20, md = run_algos(algos_oracle, n, s, d, c, hop_cap=20)
        if not (digest(M, path, e20) == golden["digest"][idx]).all() or md != int(golden["max_dist"][idx]):
            bad.append(idx)
    assert not bad, f"{len(bad)} of {G} fixture graphs differ from the reference: {bad[:10]}"


def test_restatement_matches_the_reference_golden(golden):
    """RestatedAlgos reproduces what the compiled reference produced: the hand KATs, random digraphs and sparse graphs up to
    300 nodes of the fixture, and every 20th real Gowalla-Nevada graph (the 512-node chain is left out: its walks of up to 511
    hops make the Python recursion of get_all_edges too slow for the suite)."""
    names = [str(x) for x in golden["names"]]
    checked = 0
    for idx, name in enumerate(names):
        real = name.startswith("gowalla")
        if (real and idx % 20) or int(golden["n"][idx]) > 300:
            continue
        _, n, s, d, c = golden_graph(golden, idx)
        M, path, e20, md = run_algos(RestatedAlgos, n, s, d, c, hop_cap=20)
        assert (digest(M, path, e20) == golden["digest"][idx]).all() and md == int(golden["max_dist"][idx]), name
        checked += 1
    assert checked > 400


def test_oracle_vs_compiled_reference_random():
    """Fuzz the oracle against the reference: the compiled algos.pyx when oracle/_ref is built, else its pinned restatement."""
    ref = _reference()
    rng = np.random.default_rng(5)
    for _ in range(60):
        n = int(rng.integers(1, 30))
        adj = rng.random((n, n)) < rng.choice([0.05, 0.15, 0.4])
        ef = np.zeros((n, n, 1), np.int64)
        ef[adj] = rng.integers(3, 50, size=(int(adj.sum()), 1))
        M, p = ref.floyd_warshall(adj)
        M2, p2 = algos_oracle.floyd_warshall(adj)
        assert (M == M2).all() and (p == p2).all()
        e = ref.gen_edge_input(int(M.max()), p, ef)
        e2 = algos_oracle.gen_edge_input(int(M.max()), p2, ef)
        assert e.shape == e2.shape and (e == e2).all()


def test_oracle_vs_compiled_reference_node_510_collision():
    """n = 512 with node 510 as a hub: reachable pairs whose last improving intermediate is node 510 carry path == 510 and
    are skipped by the reference's gen_edge_input (algos.pyx:87-88), while inside get_all_edges node 510 is expanded like any
    other intermediate.  The oracle must reproduce that (reference as in the random test above)."""
    ref = _reference()
    rng = np.random.default_rng(1022)
    n = 512
    adj = rng.random((n, n)) < 0.003
    adj[510, rng.random(n) < 0.3] = True
    adj[rng.random(n) < 0.3, 510] = True
    ef = np.zeros((n, n, 1), np.int64)
    ef[adj] = rng.integers(3, 50, size=(int(adj.sum()), 1))
    M, p = ref.floyd_warshall(adj)
    M2, p2 = algos_oracle.floyd_warshall(adj)
    assert (M == M2).all() and (p == p2).all()
    assert ((p == 510) & (M < 510)).sum() > 100
    md = int(M[M < 510].max())              # hop axis just long enough for every walk (keeps the reference's temp small)
    e = ref.gen_edge_input(md, p, ef)
    e2 = algos_oracle.gen_edge_input(md, p2, ef)
    assert e.shape == e2.shape and (e == e2).all()


def test_fw_invariants_property():
    """SURVEY.md §4 property checks on the oracle."""
    rng = np.random.default_rng(11)
    for _ in range(40):
        n = int(rng.integers(1, 50))
        adj = rng.random((n, n)) < 0.1
        M, p = algos_oracle.floyd_warshall(adj)
        assert (np.diag(M) == 0).all() and M.max() <= 510
        assert ((p == 510) == (M == 510)).all()
        ef = np.zeros((n, n, 1), np.int64)
        ef[adj] = 5
        md = int(M.max())
        e = algos_oracle.gen_edge_input(md, p, ef)[..., 0]
        if e.shape[-1] == 0:
            continue
        hops = (e != -1).sum(-1)
        assert (hops <= M).all()                      # the node-0 quirk can only shorten the walk
        # -1 only after the walk: once a hop is -1 all later hops are -1
        first_neg = np.where((e == -1).any(-1), (e == -1).argmax(-1), e.shape[-1])
        assert (first_neg == hops).all()
