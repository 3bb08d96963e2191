"""CPU: mobgt_b200.owndata — the reference's on-disk data set format (train.pickle / *_idx.pkl / Graph_*.csv) -> raw items and
dataset tables (SURVEY.md §8f #3), on the REAL Gowalla-Nevada data set the reference ships.

tests/golden/gowalla_nevda_real.npz was written by tests/golden/make_gowalla_real.py, which ran the UNMODIFIED reference
`owndata.GowallaGraph.process` and `model_fqandtoyo.calculate_laplacian_matrix` on the unpacked archive, compared every item
field and every matrix entry with this package's adapter, and stored sha256 digests of the REFERENCE's outputs."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(HERE, "golden"))
NPZ = os.path.join(HERE, "golden", "gowalla_nevda_real.npz")


@pytest.fixture(scope="module")
def real():
    from mobgt_b200 import owndata
    z = np.load(NPZ)
    world, splits = owndata.unpack_dataset(z)
    return z, world, splits


def test_fixture_equals_the_reference_outputs(real):
    """The unpacked fixture reproduces the digests of what the reference's own dataset code produced."""
    import _gowalla
    z, world, splits = real
    assert (world.P, world.C, world.U) == (3679, 253, 1080)
    assert len(splits["train"]) == 4970 and len(splits["test"]) == 1899            # SURVEY.md §8c
    assert _gowalla.items_digest(splits["train"]) == str(z["ref_digest_train"])
    assert _gowalla.items_digest(splits["test"]) == str(z["ref_digest_test"])
    assert _gowalla.csr_dense_digest(world.D_A, world.P) == str(z["ref_digest_D_A"])
    assert _gowalla.csr_dense_digest(world.C_A, world.C) == str(z["ref_digest_C_A"])
    # \hat A = (D + I)^-1 (A + I): every row sums to 1, the diagonal is present
    for crow, col, val in (world.D_A, world.C_A):
        n = len(crow) - 1
        sums = np.add.reduceat(val.astype(np.float64), crow[:-1])
        assert np.allclose(sums, 1.0, atol=1e-5)
        assert all(r in col[crow[r]:crow[r + 1]] for r in range(0, n, 97))
    # X = [check_freq | one-hot category | lat | lon]  (model_fqandtoyo.py:680-692)
    assert world.X.shape == (3679, 3 + 253) and np.array_equal(world.X[:, 1:254].sum(1), np.ones(3679, np.float32))
    assert np.array_equal(world.X[np.arange(3679), world.cat_of_poi], np.ones(3679, np.float32))


def test_generate_queue_orders():
    """owndata.py:60-85 on a small split: 'normal' keeps dict / list order; 'random' takes, per round, the next session of the
    first int(0.01 * users) + 1 users of a fresh shuffle (legacy generator seeded with 1) until every queue is empty."""
    from mobgt_b200 import owndata
    idx = {u: list(range(u % 3 + 1)) for u in range(7)}
    assert owndata.generate_queue(idx, "normal") == [(u, s) for u in range(7) for s in idx[u]]
    q = owndata.generate_queue(idx, "random", seed=1)
    assert sorted(q) == sorted((u, s) for u in range(7) for s in idx[u])
    for u in range(7):                                       # a user's sessions stay in order
        assert [s for (v, s) in q if v == u] == idx[u]
    rng = np.random.RandomState(1)                           # int(0.01 * 7) = 0 -> ONE user per round: the head of each shuffle
    users, left, exp = list(range(7)), {u: list(v) for u, v in idx.items()}, []
    while any(left.values()):
        rng.shuffle(users)
        if left[users[0]]:
            exp.append((users[0], left[users[0]].pop(0)))
    assert q == exp


def test_adapter_reads_files_in_the_reference_format(real, tmp_path):
    """load_world / load_items on a small data set written in the reference's on-disk format (Graph_*.csv with one header row,
    {split}.pickle = {user: {session: dict of torch tensors}}, {split}_idx.pkl = {user: [session, ...]}): the world is known by
    construction, and the items are real trajectories of the committed fixture, read back field for field."""
    import pickle
    import torch
    from mobgt_b200 import owndata
    raw = tmp_path / "raw"
    raw.mkdir()
    P, C = 6, 3
    cat = np.array([2, 1, 3, 1, 2, 3])
    poi = [(i + 1, 10 * i + 1, 36.0 + 0.25 * i, -115.5 + 0.125 * i, int(cat[i])) for i in range(P)]
    rng = np.random.default_rng(4)
    A_d, A_c = (rng.random((P, P)) < 0.4).astype(np.int64), (rng.random((C, C)) < 0.5).astype(np.int64)

    def write_csv(name, rows, header):
        (raw / name).write_text(header + "\n" + "".join(",".join(str(v) for v in r) + "\n" for r in rows))

    write_csv("Graph_poi.csv", poi, "POI ID,check_freq,latitude,longitude,cat")
    write_csv("Graph_dist.csv", A_d, ",".join(str(i) for i in range(P)))
    write_csv("Graph_cat.csv", A_c, ",".join(str(i) for i in range(C)))
    w = owndata.load_world(str(raw), "gowalla_nevda")
    assert (w.P, w.C, w.U) == (P, C, 1080) and np.array_equal(w.cat_of_poi, cat)
    assert np.array_equal(w.check_freq, [r[1] for r in poi])
    assert np.array_equal(w.latlon, np.array([r[2:4] for r in poi], np.float32))
    assert np.array_equal(w.X[:, 0], [r[1] for r in poi]) and np.array_equal(w.X[np.arange(P), cat], np.ones(P, np.float32))
    for (crow, col, val), A in ((w.D_A, A_d), (w.C_A, A_c)):
        n = len(A)
        dense = np.zeros((n, n), np.float32)
        dense[np.repeat(np.arange(n), np.diff(crow)), col] = val
        hat = ((A + np.eye(n)) / (A.sum(1) + 1)[:, None]).astype(np.float32)        # (D + I)^-1 (A + I)
        assert np.allclose(dense, hat, rtol=1e-6, atol=0)

    _, _, splits = real
    src = splits["test"][:7]
    sessions = {}
    for k, it in enumerate(src):          # two sessions per user, in the order written

        adj = np.zeros((len(it.x), len(it.x)), np.int64)
        adj[it.edge_index[0], it.edge_index[1]] = it.edge_attr
        sessions.setdefault(k // 2, {})[k % 2] = dict(
            node_name=torch.from_numpy(np.asarray(it.x).reshape(-1)), edge_type=torch.from_numpy(adj),
            target=torch.from_numpy(np.asarray(it.y)), time=torch.from_numpy(np.asarray(it.time).reshape(-1)),
            time_normal=torch.from_numpy(np.asarray(it.time_normal).reshape(-1)),
            user=torch.from_numpy(np.asarray(it.user).reshape(-1)), cat=torch.from_numpy(np.asarray(it.cat).reshape(-1)))
    with open(raw / "test.pickle", "wb") as f:
        pickle.dump(sessions, f)
    with open(raw / "test_idx.pkl", "wb") as f:
        pickle.dump({u: list(s) for u, s in sessions.items()}, f)
    got = owndata.load_items(str(raw), "test")                 # 'normal' order: users, then sessions, as written
    assert len(got) == len(src)
    for a, b in zip(got, src):
        for name in ("x", "edge_index", "edge_attr", "y", "time", "time_normal", "user", "cat"):
            assert np.array_equal(np.asarray(getattr(a, name)), np.asarray(getattr(b, name))), name


def test_real_batches_pack_and_match_the_oracle_collator(real):
    """Every 256-graph batch of the real train split goes through the product's host packing (graphs of more than 512 nodes are
    dropped as collator.py:313 does; no index leaves its embedding table), and on a real batch the packed fields equal the
    oracle's restatement of wrapper.preprocess_item + collator (pinned to the reference by tests/golden/model_golden_*)."""
    import model_oracle as mo
    from mobgt_b200 import collator
    z, world, splits = real
    train = splits["train"]
    kept = 0
    for i in range(0, len(train), 256):
        hp = collator.pack_host(train[i:i + 256])
        off, shape, dts, nbytes = hp.layout["n"]
        ns = hp.buf[off:off + nbytes].view(np.dtype(dts)).reshape(shape)
        assert ns.max() <= 512
        kept += len(ns)
    big = sum(len(it.x) > 512 for it in train)
    assert kept == len(train) - big and 0 < big < 10
    items = [it for it in train[:24] if len(it.x) <= 64]
    hp = collator.pack_host(items)

    def field(name):
        off, shape, dts, nbytes = hp.layout[name]
        return hp.buf[off:off + nbytes].view(np.dtype(dts)).reshape(shape)

    ob = mo.collate([mo.preprocess_item(it, hop_cap=20) for it in items], world, multi_hop_max_dist=20, rel_pos_max=1024)
    ns, no = field("n"), field("node_off")
    B, N = len(ns), int(ns.max())
    assert tuple(ob.x.shape[:2]) == (B, N)

    def padded(flat, dtype):
        out = np.zeros((B, N), dtype)
        for gi in range(B):
            out[gi, :ns[gi]] = flat[no[gi]:no[gi + 1]]
        return out

    assert np.array_equal(padded(field("x_nodes"), np.int64), ob.x[:, :, 0].numpy())
    assert np.array_equal(padded(field("in_deg"), np.int64), ob.in_degree.numpy())
    assert np.array_equal(padded(field("out_deg"), np.int64), ob.out_degree.numpy())
    assert np.array_equal(field("user").reshape(-1), ob.user.numpy().reshape(-1))
    assert np.array_equal(field("y").reshape(-1), ob.y.numpy().reshape(-1))


def test_hat_rw_normd_csr_equals_the_dense_formula():
    """(D + I)^-1 (A + I) of calculate_laplacian_matrix(..., 'hat_rw_normd_lap_mat') (model_fqandtoyo.py:476-484), restated with
    numpy's dense inverse as the reference writes it, on random weighted / binary / empty-row adjacency matrices."""
    from mobgt_b200 import owndata
    rng = np.random.default_rng(0)
    for n, density, weighted in ((1, 0.0, False), (7, 0.3, False), (40, 0.1, True), (64, 0.0, False), (33, 0.9, True)):
        a = (rng.random((n, n)) < density).astype(np.float64)
        if weighted:
            a *= rng.integers(1, 9, size=(n, n))
        deg = np.asmatrix(np.diag(a.sum(1)))
        ident = np.asmatrix(np.identity(n))
        ref = np.asarray(np.matmul(np.linalg.matrix_power(deg + ident, -1), np.asmatrix(a) + ident)).astype(np.float32)
        crow, col, val = owndata.hat_rw_normd_csr(a)
        got = np.zeros((n, n), np.float32)
        got[np.repeat(np.arange(n), np.diff(crow)), col] = val
        assert np.array_equal(got, ref), (n, density, weighted)
        assert np.all(np.diff(crow) >= 1)                                 # the self loop is always there
