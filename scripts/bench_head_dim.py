"""The built encoder shapes against each other: the canonical 6-layer model (ffn 1024) at 8 heads x hidden_dim 128 (d = 24),
8 heads x hidden_dim 64 (d = 16) and 12 heads x hidden_dim 128 (d = 16), on the c2-dense128 and c2-natural batches of bench.py
(256 graphs, toyotagraph-shaped world of 60 000 POIs).

    python scripts/bench_head_dim.py OUT_DIR [--steps 20] [--warmup 5] [--iters 20] [--shapes 8x128,8x64,12x128]
                                     [--edge_types multi_hop,single_hop]

For every (workload, shape) it reports, as OUT_DIR/bench_head_dim.json (one JSON object) and one line per case on stdout:
  * step: ms / step and graphs / s of the replayed training step (trainer.Trainer with CUDA graphs, as bench.py times it);
  * k3: one layer's attention forward and backward (mode 2: the per-layer bf16 dS plane the training step writes), dropout on
    (p = 0.1), CUDA events around each launch with the L2 overwritten (a 256 MB buffer zeroed) before it; mean ms over --iters;
  * k2: the attention-bias build (bf16 bias, once per step) and its backward from the n_layers bf16 dS planes, same timer;
  * bytes: what one K3 launch must move at these shapes (the live bias cells and q / k / v / out / lse, plus dout / o / dq / dk /
    dv and the dS plane in the backward), the live bias bytes per layer, and the resulting GB/s;
  * the card's name and power limit, read in the same run.
--edge_types runs every case once per edge encoding (default: multi_hop only, which writes exactly the records above).  Any
other list adds to each record its edge_type and K2's index bytes (per live pair: rel_pos 2 + poi_pos 2 + the walk's hops bytes
for multi_hop, + the one feat8 byte for the direct encoding), read once by the forward and once by the backward.
The numbers are only meaningful with a GPU: without one the script stops."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import bench  # noqa: E402  (the workloads, the canonical hyper-parameters and the kernel timer of bench.py)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, plim, clk = [s.strip() for s in q[0].split(",")] if q else (torch.cuda.get_device_name(0), "unknown", "unknown")
    return dict(name=name, power_limit=plim, max_sm_clock=clk, torch_name=torch.cuda.get_device_name(0))


def k3_bytes(batch, d, H=8):
    """bytes one attention launch must read and write at this batch: live bias cells (bf16) + q, k, v (bf16) + out (bf16) + lse
    (fp32) forward; backward: bias + q, k, v, o, dout + lse + dq, dk, dv + the live dS cells (bf16 plane)."""
    n = batch.n_host.astype(np.int64) + 1
    cells = int((n * n).sum()) * H
    ntok = int(batch.tok_pos.numel())
    fwd = 2 * cells + ntok * H * d * 2 * 4 + ntok * H * 4
    bwd = 2 * cells + ntok * H * d * 2 * 5 + ntok * H * 4 + ntok * H * d * 2 * 3 + 2 * cells
    return fwd, bwd


def run_case(workload, num_heads, hidden_dim, args, flush, edge_type="multi_hop", tag=False):
    from mobgt_b200 import collator, model as M, ops
    from mobgt_b200.trainer import Trainer
    dev = torch.device("cuda")
    cfg, ds, cap, n_fixed, nbatches = bench.TRAIN_WORKLOADS[workload]
    world = bench.make_world_for(workload)
    B = args.batch
    item_sets = [bench.make_workload(workload, world, B, 0, batch_id=i) for i in range(nbatches)]
    torch.manual_seed(1)
    hp = dict(bench.HP, hidden_dim=hidden_dim, num_heads=num_heads, edge_type=edge_type)
    model = M.Graphormer(dataset_name=ds, world=world, **hp).to(dev).train()
    tr = Trainer(model, dev, 1, cuda_graph=True)
    latlon = torch.from_numpy(world.latlon).to(dev)
    ckw = dict(world=world, latlon_dev=latlon, multi_hop_max_dist=hp["multi_hop_max_dist"], rel_pos_max=1024, device=dev)
    batches = [collator.collate_packed(its, max_node=512, bucket=nbatches > 1, **ckw) for its in item_sets]
    state = dict(i=0)

    def step():
        b = batches[state["i"] % nbatches]
        state["i"] += 1
        state["loss"] = tr.train_step(b)

    for _ in range(max(args.warmup, 2 * nbatches)):
        step()
    g0 = tr.graph_steps
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / args.steps
    replays = tr.graph_steps - g0
    loss = float(state["loss"])

    # one layer's K3 at the first batch's shapes, dropout on, L2 overwritten before every launch
    b = batches[0]
    H = num_heads
    d = (hidden_dim + 64) // H
    tabs = [t.detach().float().contiguous() for t in (model.rel_pos_encoder.weight, model.poi_pos_encoder.weight,
                                                       model.edge_encoder.weight, model.edge_dis_encoder.weight.view(-1),
                                                       model.graph_token_virtual_distance.weight.view(-1))]
    direct = model.direct_edges
    k2_fwd = (lambda: ops.bias_direct_fwd_raw(b, tabs[0], tabs[1], tabs[2], tabs[4])) if direct else (lambda: ops.bias_fwd_raw(b, *tabs))
    bias = k2_fwd()
    ntok = int(b.tok_pos.numel())
    qkv = torch.randn(ntok, 3 * H * d, device=dev).to(torch.bfloat16)
    dout = torch.randn(ntok, H * d, device=dev).to(torch.bfloat16)
    dp, sd = hp["attention_dropout_rate"], 0x5DEECE66D1234567
    out, lse = ops.attn_fwd_raw(qkv, bias, b, drop_p=dp, seed=sd)
    plane = torch.empty(tuple(bias.shape), dtype=torch.bfloat16, device=dev)
    scale = model.layers[0].self_attention.scale
    t_f = bench.time_kernel(lambda: ops.attn_fwd_raw(qkv, bias, b, scale=scale, drop_p=dp, seed=sd), flush, iters=args.iters)
    t_b = bench.time_kernel(lambda: ops.attn_bwd_raw(qkv, bias, out, dout, lse, b, plane, 2, scale=scale, drop_p=dp, seed=sd),
                            flush, iters=args.iters)
    fb, bb = k3_bytes(b, d, H)
    # K2 at the same batch: the forward writes the bf16 bias, the backward sums the n_layers bf16 dS planes
    planes = torch.randn((hp["n_layers"],) + tuple(bias.shape), device=dev).to(torch.bfloat16)
    bins = tabs[1].shape[0]
    t_k2f = bench.time_kernel(k2_fwd, flush, iters=args.iters)
    k2_bwd = (lambda: ops.bias_direct_bwd_raw(b, planes, bins)) if direct else (lambda: ops.bias_bwd_raw(b, planes, tabs[2], tabs[3], bins))
    t_k2b = bench.time_kernel(k2_bwd, flush, iters=args.iters)
    n = b.n_host
    live = int(((n.astype(np.int64) + 1) ** 2).sum())
    bias_bytes = 2 * live * H                      # live bf16 bias cells of one layer (= one dS plane)
    pairs = int((n.astype(np.int64) ** 2).sum())
    index_bytes = pairs * (2 + 2 + (1 if direct else b.hops))
    extra = dict(edge_type=edge_type) if tag else {}
    k2_extra = dict(index_bytes=index_bytes) if tag else {}
    return dict(**extra,workload=workload, num_heads=H, hidden_dim=hidden_dim, head_dim=d, n_layers=hp["n_layers"], ffn_dim=hp["ffn_dim"],
                graphs_per_step=B, tokens=ntok, nodes_max=int(n.max()), nodes_median=float(np.median(n)), padded=bool(getattr(b, "padded", False)),
                step=dict(ms=ms, graphs_per_s=B * 1e3 / ms, steps=args.steps, graph_replays=replays, loss=loss),
                k3=dict(fwd_ms=t_f, bwd_ms=t_b, fwd_bytes=fb, bwd_bytes=bb, fwd_gbs=fb / t_f / 1e6, bwd_gbs=bb / t_b / 1e6,
                        iters=args.iters, dropout=dp, l2="256 MB buffer zeroed before every launch"),
                k2=dict(fwd_ms=t_k2f, bwd_ms=t_k2b, bias_bytes_per_layer=bias_bytes, bwd_planes=hp["n_layers"],
                        fwd_gbs=bias_bytes / t_k2f / 1e6, bwd_gbs=hp["n_layers"] * bias_bytes / t_k2b / 1e6, iters=args.iters,
                        l2="256 MB buffer zeroed before every launch", **k2_extra))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--workloads", default="c2-dense128,c2-natural")
    ap.add_argument("--shapes", default="8x128,8x64,12x128", help="num_heads x hidden_dim, comma-separated")
    ap.add_argument("--edge_types", default="multi_hop", help="edge encodings, comma-separated (any value but multi_hop: direct)")
    args = ap.parse_args()
    from mobgt_b200 import _C
    _C.require_cuda()
    os.makedirs(args.out_dir, exist_ok=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = dict(card=card(), cases=[])
    tag = args.edge_types != "multi_hop"
    for wl in args.workloads.split(","):
        for et in args.edge_types.split(","):
            for nh, hd in (map(int, x.split("x")) for x in args.shapes.split(",")):
                r = run_case(wl, nh, hd, args, flush, et, tag)
                res["cases"].append(r)
                print(json.dumps(dict(**({"edge_type": et} if tag else {}), workload=wl, num_heads=nh, hidden_dim=hd, step_ms=round(r["step"]["ms"], 3),
                                      graphs_per_s=round(r["step"]["graphs_per_s"], 1), k3_fwd_ms=round(r["k3"]["fwd_ms"], 4),
                                      k3_bwd_ms=round(r["k3"]["bwd_ms"], 4), k2_fwd_ms=round(r["k2"]["fwd_ms"], 4),
                                      k2_bwd_ms=round(r["k2"]["bwd_ms"], 4), bias_mb=round(r["k2"]["bias_bytes_per_layer"] / 1e6, 2))),
                      flush=True)
    with open(os.path.join(args.out_dir, "bench_head_dim.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
