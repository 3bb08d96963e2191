"""The fp32 evaluation head (mobgt_head_topk_f32, `--precision 32`) against the bf16 head (mobgt_head_topk, `--precision 16`)
on the same inputs, at the two evaluation shapes of bench.py:
  * c2: M = 256 rows, V = 60 001 POIs, K = 320, k = 20;
  * c5 shard: M = 4 096 rows against one GPU's 125 000-row vocabulary shard, K = 320, k = 10.

    python scripts/bench_head_f32.py OUT_DIR [--iters 20]

For each shape and head it reports, as OUT_DIR/bench_head_f32.json and one line per case on stdout:
  * mode 1 + merge (the top-k lists and rank counts of every row, merged: what ops.head_topk_local runs once s_t is known) and
    mode 0 (s_t alone), in ms: CUDA events around each launch, the L2 overwritten (a 256 MB buffer zeroed) before it, mean over
    --iters after 2 warm-up calls;
  * the achieved FLOP/s of mode 1 + merge from 2 M V K;
  * the split count (lists per row) the head used;
  * how many target ranks and top-k id lists differ between the two heads on these inputs (z = ELU(LayerNorm(randn)), W and
    bias as nn.Linear initialises them: the bf16 head rounds z and W to bf16);
and the card's name and power limit, read in the same run.  The numbers are only meaningful with a GPU: without one the
script stops."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import bench  # noqa: E402  (the kernel timer of bench.py)

SHAPES = (("c2", 256, 60001, 320, 20), ("c5_shard", 4096, 125000, 320, 10))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, plim, clk = [s.strip() for s in q[0].split(",")] if q else (torch.cuda.get_device_name(0), "unknown", "unknown")
    return dict(name=name, power_limit=plim, max_sm_clock=clk, torch_name=torch.cuda.get_device_name(0))


def inputs(M, V, K, dev):
    g = torch.Generator(device=dev).manual_seed(5)
    z = torch.nn.functional.elu(torch.nn.functional.layer_norm(torch.randn(M, K, device=dev, generator=g), (K,))).contiguous()
    W = ((torch.rand(V, K, device=dev, generator=g) * 2 - 1) / K ** 0.5).contiguous()
    b = ((torch.rand(V, device=dev, generator=g) * 2 - 1) / K ** 0.5).contiguous()
    t = torch.randint(0, V, (M,), device=dev, generator=g).int()
    return z, W, b, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_head_f32.py measures on the GPU; no CUDA device is available")
    from mobgt_b200 import _C, ops
    _C.require_cuda()
    dev = torch.device("cuda")
    info = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    res = dict(card=info, iters=args.iters, timer="CUDA events per launch, L2 overwritten (256 MB zeroed) before each", cases=[])
    for name, M, V, K, k in SHAPES:
        z, W, b, t = inputs(M, V, K, dev)
        heads = {"fp32": (z, W), "bf16": (z.to(torch.bfloat16), W.to(torch.bfloat16))}
        outs = {}
        for head, (zh, Wh) in heads.items():
            st = ops.head_target_logit(zh, Wh, b, t)
            t1 = bench.time_kernel(lambda: ops.head_topk_local(zh, Wh, b, t, k, st=st), flush, iters=args.iters)
            t0 = bench.time_kernel(lambda: ops.head_target_logit(zh, Wh, b, t), flush, iters=args.iters)
            outs[head] = ops.head_topk_local(zh, Wh, b, t, k, st=st)
            flop = 2.0 * M * V * K
            rec = dict(shape=name, head=head, M=M, V=V, K=K, k=k, nsplit=ops.head_split(M, V, zh.dtype), mode1_merge_ms=round(t1, 4),
                       mode0_ms=round(t0, 4), tflops_mode1=round(flop / (t1 * 1e-3) / 1e12, 2))
            res["cases"].append(rec)
            print(json.dumps(rec), flush=True)
        f, h = outs["fp32"], outs["bf16"]
        dr = (f["cnt"].long() - h["cnt"].long()).abs()
        diff = dict(shape=name, ranks_differing=int((dr > 0).sum()), mean_abs_rank_shift=round(float(dr.double().mean()), 2),
                    max_abs_rank_shift=int(dr.max()), topk_lists_differing=int((f["idx"] != h["idx"]).any(1).sum()), rows=M)
        res.setdefault("fp32_vs_bf16", []).append(diff)
        print(json.dumps(diff), flush=True)
        del z, W, heads, outs
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "bench_head_f32.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(info))


if __name__ == "__main__":
    main()
