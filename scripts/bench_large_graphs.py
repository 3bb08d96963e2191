"""Cost of graphs of 513 to 1 024 nodes (T = 514 .. 1 025 tokens) on the model path.

    python scripts/bench_large_graphs.py [--iters 20] [--out profiles/large_graphs/bench_large_graphs.json]

Records, on the GPU it runs on:
  * the card's name, power limit and max SM clock, read in the same run;
  * K2 (attention-bias build, multi-hop, 8 heads, hops 20, bf16 plane) forward / backward (6 bf16 dS planes) and K3 (bf16
    attention, head dim 24, dropout 0.1) forward / backward (mode 2) on a batch of ONE synthetic trajectory graph of
    T - 1 nodes, T = 627, 815, 1 025: CUDA events around each launch with the L2 overwritten (a 256 MB buffer zeroed) before it,
    mean ms over --iters;
  * the eager training-step time (forward + backward + AdamW, MobGT 6 layers x 8 heads x 128, bf16) of a real Gowalla-Nevada
    batch of 256 train trajectories holding the 814-node one, against the same batch without it (255 trajectories); the two
    are timed alternately, --iters steps each after a warm-up.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, plim, clk = [s.strip() for s in q[0].split(",")] if q else ("?", "?", "?")
    return dict(name=name, power_limit=plim, max_sm_clock=clk, torch_name=torch.cuda.get_device_name(0))


def timed(fn, iters, flush):
    """mean ms of fn() over iters launches, the L2 overwritten before each"""
    ts = []
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.mean(ts)), float(np.std(ts))


def kernels(T, iters, flush):
    from mobgt_b200 import collator, ops, synth
    w = synth.make_world("c4", seed=1)
    items = synth.make_items(w, 1, T - 1, seed=T, n_fixed=T - 1)
    b = collator.collator_gowalla(items, max_node=1024, multi_hop_max_dist=20, rel_pos_max=1024, world=w, large_graphs=True)
    assert b.N + 1 == T
    H, d, bins = 8, 24, int(w.num_bins)
    g = torch.Generator(device="cuda").manual_seed(T)
    R, Pp, E = (torch.randn(r, H, device="cuda", generator=g) * 0.3 for r in (512, bins, 128))
    W = torch.randn(128 * H * H, device="cuda", generator=g) * 0.3
    tvd = torch.randn(H, device="cuda", generator=g) * 0.3
    bias = ops.bias_fwd_raw(b, R, Pp, E, W, tvd, out_dtype=torch.bfloat16)
    planes = torch.randn((6,) + tuple(bias.shape), device="cuda", generator=g).to(torch.bfloat16)
    ntok = int(b.tok_pos.numel())
    qkv = (torch.randn(ntok, 3 * H * d, device="cuda", generator=g)).to(torch.bfloat16)
    dout = torch.randn(ntok, H * d, device="cuda", generator=g).to(torch.bfloat16)
    out, lse = ops.attn_fwd_raw(qkv, bias, b, drop_p=0.1, seed=5)
    ds = torch.empty(bias.shape, dtype=torch.bfloat16, device="cuda")
    fns = dict(k2_fwd=lambda: ops.bias_fwd_raw(b, R, Pp, E, W, tvd, out_dtype=torch.bfloat16),
               k2_bwd=lambda: ops.bias_bwd_raw(b, planes, E, W, bins),
               k3_fwd=lambda: ops.attn_fwd_raw(qkv, bias, b, drop_p=0.1, seed=5),
               k3_bwd=lambda: ops.attn_bwd_raw(qkv, bias, out, dout, lse, b, ds, 2, drop_p=0.1, seed=5))
    res = {}
    for k, fn in fns.items():
        fn()
        torch.cuda.synchronize()
        m, s = timed(fn, iters, flush)
        res[k] = dict(ms=round(m, 4), std=round(s, 4))
    return res


def steps(iters):
    from mobgt_b200 import collator, model, owndata
    from mobgt_b200.trainer import Trainer
    world, splits = owndata.unpack_dataset(np.load(os.path.join(ROOT, "tests", "golden", "gowalla_nevda_real.npz")))
    tr_items = splits["train"]
    big = [i for i, it in enumerate(tr_items) if len(it.x) == 814][0]
    ordinary = [it for it in tr_items if len(it.x) <= 512][:255]
    with_big = ordinary + [tr_items[big]]
    hp = dict(n_layers=6, num_heads=8, hidden_dim=128, dropout_rate=0.1, intput_dropout_rate=0.1, weight_decay=0.01, ffn_dim=1024,
              warmup_updates=40000, tot_updates=400000, peak_lr=2e-4, end_lr=1e-9, edge_type="multi_hop", multi_hop_max_dist=20,
              attention_dropout_rate=0.1)
    torch.manual_seed(1)
    m = model.Graphormer(dataset_name="gowalla_nevda", world=world, precision=16, **hp).cuda().train()
    tr = Trainer(m, torch.device("cuda"), cuda_graph=False)
    kw = dict(max_node=1024, multi_hop_max_dist=20, rel_pos_max=1024, world=world, large_graphs=True)
    batches = dict(with_814=collator.collator_gowalla(with_big, **kw), without_814=collator.collator_gowalla(ordinary, **kw))
    assert batches["with_814"].N == 814 and batches["without_814"].N <= 512
    ts = {k: [] for k in batches}
    for k, b in batches.items():                       # warm-up
        for _ in range(2):
            tr.train_step(b)
    torch.cuda.synchronize()
    for _ in range(iters):
        for k, b in batches.items():
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            tr.train_step(b)
            e.record()
            torch.cuda.synchronize()
            ts[k].append(a.elapsed_time(e))
    res = {k: dict(ms=round(float(np.mean(v)), 3), std=round(float(np.std(v)), 3), graphs=int(batches[k].B), N=int(batches[k].N))
           for k, v in ts.items()}
    res["ratio"] = round(res["with_814"]["ms"] / res["without_814"]["ms"], 3)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "large_graphs", "bench_large_graphs.json"))
    args = ap.parse_args()
    from mobgt_b200 import _C
    _C.require_cuda()
    torch.cuda.set_device(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = dict(card=card(), kernels={str(T): kernels(T, args.iters, flush) for T in (627, 815, 1025)}, step=steps(args.iters))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
