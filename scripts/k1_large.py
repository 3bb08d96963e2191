"""K1 on graphs of 513..1024 nodes (k1_apsp_large_kernel + k1_walk_from_path_kernel) against the C oracle on the host.

    python scripts/k1_large.py [OUT_DIR] [--iters 5]        (default OUT_DIR: profiles/k1_large)

Cases:
  * the two train trajectories of the shipped Gowalla-Nevada data set above 512 nodes (626 and 814 nodes), through the per-item
    drop-in as wrapper.py:55-60 calls it: floyd_warshall, then gen_edge_input at the full max_dist (510 and 85 hop slots).
    Reported: the device time of its two K1 calls (mobgt_apsp_edge_input with `path`, mobgt_gen_edge_input), CUDA events with
    the inputs resident, and the host wall time of the two Python calls (copies and the float32 [n, n, max_dist, 1] array
    included);
  * synthetic 1024-node graphs (random, ~2 out-edges per node), 1, 16 and 64 per launch, through apsp_edge_input_packed with
    20 hop slots: Floyd-Warshall alone (want_edges=False) and Floyd-Warshall + walk.
Device times: CUDA events around each call, the L2 overwritten (256 MB zeroed) before it, mean over --iters after 2 warm-up
calls.  Next to them: the C oracle (oracle/algos_oracle.c, -O2, one host core) on the same graphs — for the 16 / 64-graph
launches timed on the first 4 graphs and scaled — the cluster size of the plan at each n, and the card's name and power limit,
read in the same run.  Writes OUT_DIR/k1_large.json.  The numbers are only meaningful with a GPU: without one the script stops."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "scripts")):
    sys.path.insert(0, p)
sys.dont_write_bytecode = True

import bench  # noqa: E402  (the kernel timer of bench.py)
from bench_head_f32 import card  # noqa: E402

REAL = ((1559, 626), (1589, 814))      # train-split index, node count


def cluster_size(n):
    """The cluster the n > 512 plan of csrc/k1_apsp.cu picks (pick_cluster_large): the smallest of 8 / 16 CTAs whose M slice
    (n x W u16, W = ceil(n / C) rounded up to 8) and colM[2][n8] fit 227 KB."""
    def round_up(a, b):
        return (a + b - 1) // b * b

    for C in (8, 16):
        W = round_up((n + C - 1) // C, 8)
        smem = n * W * 2 + 2 * round_up(n, 8) * 2 + 16
        if smem <= 227 * 1024:
            return dict(C=C, W=W, smem_bytes=smem)
    return None


def oracle_time(adj, ef, hop_cap):
    import algos_oracle
    t = time.perf_counter()
    M, path = algos_oracle.floyd_warshall(adj)
    algos_oracle.gen_edge_input(int(M.max()), path, ef, hop_cap=hop_cap)
    return time.perf_counter() - t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir", nargs="?", default=os.path.join(ROOT, "profiles", "k1_large"))
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("k1_large.py measures on the GPU; no CUDA device is available")
    from mobgt_b200 import _C, algos, owndata
    from mobgt_b200.algos import apsp_edge_input_packed, pack_graphs
    _C.require_cuda()
    dev = torch.device("cuda")
    info = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    res = dict(card=info, iters=args.iters, timer="CUDA events per call, L2 overwritten (256 MB zeroed) before each",
               plans={n: cluster_size(n) for n in (513, 626, 814, 880, 1024)}, cases=[])

    _, splits = owndata.unpack_dataset(np.load(os.path.join(ROOT, "tests", "golden", "gowalla_nevda_real.npz")))
    for idx, n in REAL:
        it = splits["train"][idx]
        assert len(it.x) == n
        ei = np.asarray(it.edge_index)
        adj = np.zeros((n, n), bool)
        adj[ei[0], ei[1]] = True
        ef = np.zeros((n, n, 1), np.int64)
        ef[ei[0], ei[1], 0] = np.asarray(it.edge_attr).reshape(-1) + 2          # attn_edge_type, wrapper.py:49-53
        algos.gen_edge_input(4, algos.floyd_warshall(adj[:600, :600])[1], ef[:600, :600])     # warm-up: module load, allocator
        t = time.perf_counter()
        M, path = algos.floyd_warshall(adj)
        md = int(M.max())
        e = algos.gen_edge_input(md, path, ef)
        wall = time.perf_counter() - t
        del e
        feat = torch.from_numpy(np.ascontiguousarray(adj, dtype=np.uint8).reshape(-1)).to(dev)
        nn_, sq, _ = pack_graphs([n])
        nd, sd = torch.from_numpy(nn_).to(dev), torch.from_numpy(sq).to(dev)
        fw_ms = bench.time_kernel(lambda: apsp_edge_input_packed(feat, nd, sd, nn_, hops=4, want_path=True, want_edges=False),
                                  flush, iters=args.iters)
        p16 = torch.from_numpy(path.astype(np.int16).reshape(-1)).to(dev)
        f8 = torch.from_numpy(ef[..., 0].astype(np.uint8).reshape(-1)).to(dev)
        eb = torch.empty((n * n, md), dtype=torch.uint8, device=dev)
        walk_ms = bench.time_kernel(lambda: _C.call("mobgt_gen_edge_input", _C.ptr(p16), _C.ptr(f8), _C.ptr(nd), _C.ptr(sd), 1, n, md,
                                                    0, _C.ptr(eb), _C.stream_ptr()), flush, iters=args.iters)
        ora = oracle_time(adj, ef, None)
        rec = dict(case=f"gowalla_train_{idx}", n=n, edges=int(adj.sum()), max_dist=md, graphs_per_launch=1,
                   plan=cluster_size(n), fw_ms=round(fw_ms, 3), walk_ms=round(walk_ms, 3), fw_walk_ms=round(fw_ms + walk_ms, 3),
                   dropin_wall_ms=round(wall * 1e3, 1), oracle_ms=round(ora * 1e3, 1))
        res["cases"].append(rec)
        print(json.dumps(rec), flush=True)
        del eb

    n, hops = 1024, 20
    rng = np.random.default_rng(1024)
    adjs = [rng.random((n, n)) < 2.0 / n for _ in range(64)]
    for a in adjs:
        np.fill_diagonal(a, False)
    feats = [np.where(a, rng.integers(2, 100, size=(n, n)), 0).astype(np.uint8) for a in adjs]
    ora = [oracle_time(a, f[..., None].astype(np.int64), hops) for a, f in zip(adjs[:4], feats[:4])]
    for G in (1, 16, 64):
        nn_, sq, _ = pack_graphs([n] * G)
        fd = torch.from_numpy(np.concatenate([f.reshape(-1) for f in feats[:G]])).to(dev)
        nd, sd = torch.from_numpy(nn_).to(dev), torch.from_numpy(sq).to(dev)
        fw_ms = bench.time_kernel(lambda: apsp_edge_input_packed(fd, nd, sd, nn_, hops, 1, want_path=True, want_edges=False), flush,
                                  iters=args.iters)
        fw_walk_ms = bench.time_kernel(lambda: apsp_edge_input_packed(fd, nd, sd, nn_, hops, 1), flush, iters=args.iters)
        rec = dict(case=f"synthetic_n1024_G{G}", n=n, graphs_per_launch=G, hops=hops, plan=cluster_size(n), fw_ms=round(fw_ms, 3),
                   fw_walk_ms=round(fw_walk_ms, 3), graphs_per_s=round(G / (fw_walk_ms * 1e-3), 1),
                   oracle_ms=round(float(np.mean(ora)) * G * 1e3, 1), oracle_ms_per_graph=round(float(np.mean(ora)) * 1e3, 1))
        res["cases"].append(rec)
        print(json.dumps(rec), flush=True)
        del fd

    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "k1_large.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(info))


if __name__ == "__main__":
    main()
