#!/usr/bin/env python
"""bench.py — MobGT hot-path throughput on N B200s, next to the reference's CPU path.

    python bench.py --gpus 1 --steps 20 --warmup 5                       # this framework (libmobgt kernels)
    python bench.py --impl reference --gpus 1 --steps K --warmup W       # the reference's CPU implementation of the path
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W                        # data parallel, one rank per GPU (weak scaling)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR     # + what the last timed step computed, as DIR/*.npy

Workloads (`--workload`, BASELINE.json configs):
  c2-dense128 (default)  configs[1]: toyotagraph-shaped world (60 000 POIs, 300 categories, 995 users), hidden 128 (+64), 8 heads,
                         6 layers, ffn 1024, multi_hop_max_dist 20, batch 256 graphs per GPU, bf16; every graph at the 128-node cap
                         (the stress variant SURVEY.md §8d quotes its byte counts on)
  c2-natural             same, node counts drawn from the real Gowalla-Nevada histogram clipped to 128; the timed steps cycle
                         through 8 DIFFERENT batches, so the shapes vary from step to step as in a real epoch
  c4-gowalla256          configs[3]: gowalla_nevda-shaped world (3 679 POIs, 253 categories), graphs <= 256 nodes (natural law),
                         GradientTailLoss, data parallel;  c4-dense256: every graph at 256 nodes (T = 257: the fold path of K3)
  c4-gowalla-real        the same model on the REAL Gowalla-Nevada data set the reference ships (gowalla_nevda.7z: 3 679 POIs,
                         4 970 train trajectories of 2 .. 512 nodes in the reference's queue order), frozen as
                         tests/golden/gowalla_nevda_real.npz by the reference's own dataset code (tests/golden/make_gowalla_real.py)
  c5-eval                configs[4]: the evaluation head over a 1 M-POI vocabulary sharded across the N GPUs, 4 096 rows per
                         step, fused GEMM + top-10 + rank (K5), all-gather / merge over NVLink; metric = eval rows / s
  c3-preprocess          configs[2]: K1 (floyd_warshall + gen_edge_input) over 100 000 graphs <= 512 nodes; metric = graphs / s
One training step = forward + loss + backward + (NCCL all-reduce) + AdamW over one batch, driven by
`mobgt_b200.trainer.Trainer` — the same class `python -m mobgt_b200.entry` runs; nothing is skipped or cached.

value  = units/s with the inputs already resident in HBM;
e2e    = units/s through the public API from HOST buffers: raw items -> collator (pack, H2D, K1 APSP + path edges on
         the GPU) -> training step -> loss read back, every step.

--dump-outputs DIR writes, after the timed steps of `value`, what the last of them computed (rank 0): for a training workload
the loss, and every parameter after the optimizer step and its gradient (`loss.npy`, `param.<name>.npy`, `grad.<name>.npy`);
for c5-eval the head's top-k values / ids, target ranks and target logits; for c3-preprocess K1's outputs of the last batch of
graphs.  The inputs are seeded, so two builds run with the same arguments can be compared array for array (see dump_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark writes nothing into the source tree: without this, importing the package modules that build() did not import
# (trainer, model, ops, ...) would add their .pyc files under mobgt_b200/__pycache__/
sys.dont_write_bytecode = True

HP = dict(n_layers=6, num_heads=8, hidden_dim=128, dropout_rate=0.1, intput_dropout_rate=0.1, weight_decay=0.01, ffn_dim=1024,
          warmup_updates=40000, tot_updates=400000, peak_lr=2e-4, end_lr=1e-9, edge_type="multi_hop", multi_hop_max_dist=20,
          attention_dropout_rate=0.1)      # README.md:62 canonical flags


_REAL_STDOUT = None


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_SAMPLE = 1 << 15            # values kept per dumped array: at most 256 KB each, a few tens of MB for a whole model
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write every array of `arrays` (name -> tensor / ndarray; None is skipped) as out_dir/<name>.npy: floating point as
    float32 (float64 stays float64), integers as float64 (exact).  An array of more than DUMP_SAMPLE values is replaced by the
    values at DUMP_SAMPLE fixed positions of its flattened form (sorted, drawn with seed 0 from its size alone), so the files of
    two runs line up value for value."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        if a is None:
            continue
        a = (a.detach() if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a))).reshape(-1)
        if a.numel() > DUMP_SAMPLE:        # sampled where the array lives: only DUMP_SAMPLE values are converted and copied
            pos = np.sort(np.random.default_rng(0).choice(a.numel(), DUMP_SAMPLE, replace=False))
            a = a[torch.from_numpy(pos).to(a.device)]
        a = (a.float() if a.is_floating_point() and a.dtype != torch.float64 else a.double()).cpu().numpy()
        total += a.nbytes
        if total > DUMP_LIMIT:
            raise RuntimeError(f"--dump-outputs: more than {DUMP_LIMIT >> 20} MB at {name}")
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc=d["bf16_tflops"], src="measured")
    return dict(hbm=6650.0, tc=1590.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        rows = [r for r in rows if len(r) >= 7]
        if not rows:
            return out
        sm = [float(r[0]) for r in rows]
        out["sm_mhz"] = float(np.median(sm))
        out["sm_max_mhz"] = float(rows[0][1])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        out["reasons"] = [n for i, n in enumerate(names) if any(r[3 + i].strip().lower().startswith("active") for r in rows)]
        out["samples"] = len(rows)
        return out


TRAIN_WORKLOADS = {
    # name: (synth config, dataset_name, node cap, fixed node count | None, distinct batches cycled through)
    "c2-dense128": ("c2", "toyotagraph", 128, 128, 1),
    "c2-natural": ("c2", "toyotagraph", 128, None, 8),
    "c4-gowalla256": ("c4", "gowalla_nevda", 256, None, 8),
    "c4-dense256": ("c4", "gowalla_nevda", 256, 256, 1),
    # the REAL Gowalla-Nevada data set the reference ships (gowalla_nevda.7z), frozen by tests/golden/make_gowalla_real.py through
    # the reference's own owndata.GowallaGraph.process / calculate_laplacian_matrix: consecutive 256-graph batches of the train
    # split in the reference's queue order (graphs of more than 512 nodes dropped, collator.py:313)
    "c4-gowalla-real": ("real", "gowalla_nevda", 512, None, 8),
}
WORLD_NOTE = {"c2": "toyotagraph-shaped P=60000 C=300 U=995", "c4": "gowalla_nevda-shaped P=3679 C=253 U=1080",
              "real": "real Gowalla-Nevada (gowalla_nevda.7z of the reference): P=3679 C=253 U=1080, 4 970 train trajectories in the "
                      "reference's queue order (tests/golden/gowalla_nevda_real.npz)"}
DATA_NOTE = {"real": "real trajectories (the reference's gowalla_nevda.7z via tests/golden/gowalla_nevda_real.npz), random-init weights"}
_REAL = {}


def real_dataset():
    """(PoiWorld, {split: items}) of the committed real-data fixture (mobgt_b200.owndata.unpack_dataset)."""
    if not _REAL:
        from mobgt_b200 import owndata
        world, splits = owndata.unpack_dataset(np.load(os.path.join(ROOT, "tests", "golden", "gowalla_nevda_real.npz")))
        _REAL.update(world=world, splits={k: [it for it in v if len(it.x) <= 512] for k, v in splits.items()})
    return _REAL["world"], _REAL["splits"]


def make_world_for(workload):
    from mobgt_b200 import synth
    cfg, ds, _, _, _ = TRAIN_WORKLOADS[workload]
    if cfg == "real":
        return real_dataset()[0]
    return synth.make_world(cfg, seed=1, dataset_name=ds)


def make_workload(workload, world, B, rank, seed=1, batch_id=0):
    """The raw items of batch `batch_id` of rank `rank` (disjoint across ranks and batches)."""
    from mobgt_b200 import synth
    cfg, _, cap, n_fixed, nb = TRAIN_WORKLOADS[workload]
    if cfg == "real":                 # 19 batches of 256 in the split: ranks / batches past the end wrap around
        items = real_dataset()[1]["train"]
        start = (rank * nb + batch_id) * B
        return [items[(start + j) % len(items)] for j in range(B)]
    return synth.make_items(world, B, cap, seed=seed, cfg_id=2 if cfg == "c2" else 4, n_fixed=n_fixed,
                            start=(rank * nb + batch_id) * B)


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
_PRE = {}     # state inherited by the forked preprocessing workers


def _pre_worker(i):
    """One DataLoader-worker's share (data.py:255-267, wrapper.py:25-102): the reference's preprocess_item on raw item i with
    the compiled algos.pyx (oracle/_ref) when present, else the C port — full cost, the 510-deep hop axis included
    (wrapper.py:58-60); the hop axis is sliced to multi_hop_max_dist before it crosses the process boundary, as the
    collator does inside the reference's worker (collator.py:323)."""
    mo, algos_oracle, ref_algos = _PRE["mo"], _PRE["algos_oracle"], _PRE["ref"]
    if ref_algos is not None:
        algos_oracle.floyd_warshall = ref_algos.floyd_warshall
        algos_oracle.gen_edge_input = lambda md, p, ef, hop_cap=None: ref_algos.gen_edge_input(md, p, ef)
    it = mo.preprocess_item(_PRE["items"][i], hop_cap=None)
    it.edge_input = it.edge_input[:, :, :20].contiguous()
    return {k: (v.numpy() if isinstance(v, torch.Tensor) else v) for k, v in it.__dict__.items()}


def _pre_init():
    torch.set_num_threads(1)


def cpu_reference_rate(workload, steps, warmup, full_batch=256):
    """The reference's own CPU implementation of the path on the host cores, on the SAME workload and batch size:
      * preprocessing: compiled algos.pyx (oracle/_ref; else the C port) driven like wrapper.py:55-60, in min(8, cores)
        worker processes (README.md:62 `--num_workers 8`);
      * collator + model_fqandtoyo restatement (oracle/model_oracle.py): forward + loss + backward + AdamW, all torch threads.
    A full 256-graph step takes minutes on the CPU, so each timed step runs a bounded SAMPLE of S graphs, alternating between
    two sizes S1 < S2; step time is fitted as F + S*g (F: per-step fixed cost — GCN tables over all POIs, the head over the
    whole vocabulary, AdamW over all parameters; g: per-graph cost) and the reported rate is the FULL batch extrapolated:
    value = B / (F + B*g).  Both raw timings are returned."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import multiprocessing as mp
    import algos_oracle
    import build_ref
    import model_oracle as mo
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref_algos = build_ref.load()
    cfg, ds, cap, n_fixed, _ = TRAIN_WORKLOADS[workload]
    world = make_world_for(workload)
    big = (n_fixed or 0) >= 128
    S1, S2 = (4, 12) if big else (32, 96)
    items = make_workload(workload, world, S2, 0)
    torch.manual_seed(1)
    model = mo.Graphormer(world, n_layers=HP["n_layers"], ffn_dim=HP["ffn_dim"], dropout_rate=HP["dropout_rate"],
                          intput_dropout_rate=HP["intput_dropout_rate"], attention_dropout_rate=HP["attention_dropout_rate"],
                          pos_dropout=0.1, dataset_name=ds).train()
    opt = torch.optim.AdamW(model.parameters(), lr=HP["peak_lr"], weight_decay=HP["weight_decay"])
    workers = min(8, cores)
    _PRE.update(mo=mo, algos_oracle=algos_oracle, ref=ref_algos, items=items)
    pool = mp.get_context("fork").Pool(workers, initializer=_pre_init)

    def step(S):
        t0 = time.perf_counter()
        pre = [mo.Item(**{k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in d.items()})
               for d in pool.map(_pre_worker, range(S), chunksize=max(1, S // (4 * workers)))]
        t1 = time.perf_counter()
        b = mo.collate(pre, world, multi_hop_max_dist=20, rel_pos_max=1024)
        loss = model.training_loss(b)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return time.perf_counter() - t0, t1 - t0

    try:
        for i in range(warmup):
            step(S1 if i % 2 == 0 else S2)
        ts = {S1: [], S2: []}
        tp = {S1: [], S2: []}
        t0 = time.perf_counter()
        for i in range(steps):
            S = S1 if i % 2 == 0 else S2
            dt, dpre = step(S)
            ts[S].append(dt)
            tp[S].append(dpre)
        wall = time.perf_counter() - t0
    finally:
        pool.terminate()
    m1 = float(np.mean(ts[S1]))
    m2 = float(np.mean(ts[S2])) if ts[S2] else m1 * S2 / S1
    g = max((m2 - m1) / (S2 - S1), 1e-9)
    F = max(m1 - S1 * g, 0.0)
    full = F + full_batch * g
    graphs_done = sum(len(v) * k for k, v in ts.items())
    return dict(value=full_batch / full, ms_per_step=1e3 * full, cores=cores, workers=workers, S=(S1, S2),
                step_s=(m1, m2), pre_s=(float(np.mean(tp[S1])), float(np.mean(tp[S2])) if tp[S2] else None),
                fixed_s=F, per_graph_s=g, sampled_rate=graphs_done / wall, full_batch=full_batch,
                algos="reference (compiled algos.pyx, oracle/_ref)" if ref_algos is not None else "port (oracle/algos_oracle.c)")


def _cpu_sample_text(r, steps, warm):
    return (f"{steps} timed steps after {warm} warm-up, alternating samples of {r['S'][0]} / {r['S'][1]} graphs of the same "
            f"workload: {r['step_s'][0]:.2f} s / {r['step_s'][1]:.2f} s per step -> fixed {r['fixed_s']:.2f} s + {r['per_graph_s'] * 1e3:.1f} ms/graph; "
            f"value = the full {r['full_batch']}-graph step extrapolated, {r['full_batch']} / (F + {r['full_batch']} g) "
            f"(raw sampled rate {r['sampled_rate']:.2f} graphs/s); preprocessing = {r['algos']} in {r['workers']} worker "
            f"processes, collator + model_fqandtoyo = CPU restatement (oracle/model_oracle.py), fwd+bwd+AdamW, {r['cores']} torch threads")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "c3-preprocess":
        return run_c3_reference(args)
    if args.workload == "c5-eval":
        return run_c5_reference(args)
    steps, warm = max(1, args.steps), max(1, args.warmup)
    r = cpu_reference_rate(args.workload, steps, warm, full_batch=args.batch)
    cfg = TRAIN_WORKLOADS[args.workload][0]
    line = {"metric": "train_graphs_per_sec", "value": r["value"], "unit": "graphs/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": DATA_NOTE.get(cfg, "synthetic"), "impl": "reference",
            "config": {"workload": args.workload, "world": WORLD_NOTE[cfg], "hidden": 128, "layers": 6,
                       "heads": 8, "ffn": 1024, "multi_hop_max_dist": 20, "graphs_per_gpu": args.batch},
            "cpu_baseline": {"value": r["value"], "unit": "graphs/s", "cores": r["cores"], "kind": "port",
                             "parts": {"algos": r["algos"], "collator+model": "port (oracle/model_oracle.py)"},
                             "sample": _cpu_sample_text(r, steps, warm)},
            "e2e": {"value": r["value"], "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------------ kernel micro-timing
def time_kernel(fn, flush, iters=8, warm=2):
    """CUDA-event time of fn() on the current stream, L2 flushed before every launch; returns mean ms."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for _ in range(warm):
        fn()
    for a, b in ev:
        flush.zero_()
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.mean([a.elapsed_time(b) for a, b in ev]))


def kernel_report(model, batch, pk, iters=8, head_c5=True):
    """Per-kernel device time at the workload's shapes + algorithmic bytes (SURVEY.md §8d, DESIGN.md) -> roofline."""
    import torch.nn.functional as F_
    from mobgt_b200 import ops
    from mobgt_b200.algos import apsp_edge_input_packed
    dev = torch.device("cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    B, H, T = batch.B, 8, batch.N + 1
    Tp = ops.bias_pitch(T)
    n = batch.n_host.astype(np.int64)
    cells, pairs_t, ntok = int((n * n).sum()), int(((n + 1) ** 2).sum()), int(batch.tok_pos.numel())
    hops, dk = batch.hops, int(getattr(batch, "dk", batch.hops))
    tabs = [t.detach().float().contiguous() for t in (model.rel_pos_encoder.weight, model.poi_pos_encoder.weight,
                                                       model.edge_encoder.weight, model.edge_dis_encoder.weight.view(-1),
                                                       model.graph_token_virtual_distance.weight.view(-1))]
    bias = ops.bias_fwd_raw(batch, *tabs)
    qkv = torch.randn(ntok, 576, device=dev).to(torch.bfloat16)
    dp, ds = HP["attention_dropout_rate"], 0x5DEECE66D1234567      # K3 is timed as the training step runs it: dropout on
    out, lse = ops.attn_fwd_raw(qkv, bias, batch, drop_p=dp, seed=ds)
    dout = torch.randn(ntok, 192, device=dev).to(torch.bfloat16)
    n_layers = len(model.layers)
    planes = torch.zeros((n_layers,) + tuple(bias.shape), dtype=torch.bfloat16, device=dev)   # per-layer dS planes (bf16)
    rep = {}
    tk = lambda fn: time_kernel(fn, flush, iters=iters, warm=min(2, iters))

    def add(name, ms, nbytes, per_step, flops=None):
        rep[name] = dict(ms=ms, gbs=nbytes / ms / 1e6, frac_hbm=nbytes / ms / 1e6 / pk["hbm"], bytes=nbytes, launches_per_step=per_step)
        if flops:
            rep[name]["tflops"] = flops / ms / 1e9
            rep[name]["frac_tc"] = flops / ms / 1e9 / pk["tc"]

    add("k1_apsp_edge_input", tk(lambda: apsp_edge_input_packed(batch.feat8, batch.n, batch.sq_off, batch.n_host, hops, 1, dk=dk)),
        cells * (1 + 2 + hops), 0)
    # K1's second roofline (SURVEY.md §8d "report both"): 2 n^3 u16 min-plus ops per graph against the alu-pipe peak of packed
    # u16x2 instructions: 148 SMs x 4 SMSPs x 16 lanes/clk x 2 halves x 1.965 GHz = 37.2 T op/s
    int_peak = 148 * 4 * 16 * 2 * 1.965e9 / 1e12
    rep["k1_apsp_edge_input"]["int_alu_T_ops"] = float((2.0 * n.astype(np.float64) ** 3).sum()) / rep["k1_apsp_edge_input"]["ms"] / 1e9
    rep["k1_apsp_edge_input"]["frac_int_alu"] = rep["k1_apsp_edge_input"]["int_alu_T_ops"] / int_peak
    add("k2_bias_fwd", tk(lambda: ops.bias_fwd_raw(batch, *tabs)), cells * (4 + hops) + H * pairs_t * 2, 1)
    add("k2_bias_bwd", tk(lambda: ops.bias_bwd_raw(batch, planes, tabs[2], tabs[3], tabs[1].shape[0])),
        cells * (4 + hops) + n_layers * H * pairs_t * 2, 1)
    fl = 4.0 * H * pairs_t * 24
    add("k3_attn_fwd", tk(lambda: ops.attn_fwd_raw(qkv, bias, batch, drop_p=dp, seed=ds)), 4 * ntok * 192 * 2 + H * pairs_t * 2, 6, fl)
    add("k3_attn_bwd", tk(lambda: ops.attn_bwd_raw(qkv, bias, out, dout, lse, batch, planes[0], 2, drop_p=dp, seed=ds)),
        8 * ntok * 192 * 2 + H * pairs_t * 2 + H * pairs_t * 2, 6, 2.5 * fl)
    Gd, Gc = model.gcn_tables()
    Gd, Gc = Gd.detach(), Gc.detach()
    Tm = model.time_embed_model_48.weight.detach()
    nn_ = ntok - B
    add("k4_embed_gather", tk(lambda: ops.embed_gather_raw(batch, model.cat_of_poi, Gd, Tm, Gc)),
        nn_ * (192 * 4 + 192 * 2 + 12), 1)
    nf = torch.randn(nn_, 192, device=dev).to(torch.bfloat16)
    pe, gt = model.pos_embed.pe.detach(), model.graph_token.weight.detach().view(-1)
    Din, Dout = model.in_degree_encoder.weight.detach(), model.out_degree_encoder.weight.detach()
    add("k4_embed_sum", tk(lambda: ops.embed_sum_raw(batch, nf, Din, Dout, pe, gt)),
        nn_ * (192 * 2 + 3 * 192 * 4 + 16) + ntok * 192 * 2, 1)
    g = torch.randn(ntok, 192, device=dev).to(torch.bfloat16)
    plan = ops.sort_plan(batch.tok_pos)
    add("k4_segment_sum", tk(lambda: ops.segment_sum_raw(g, 0, 192, plan, 2000)), ntok * (192 * 2 + 8), 6)
    # K6 — encoder row ops (SURVEY §8f #2, first slice): LayerNorm fwd / bwd at [ntok, 192], bias-gradient column sums
    ln = model.layers[0].ffn_norm2
    xs = torch.randn(ntok, 192, device=dev)
    dy32, dy16 = torch.randn(ntok, 192, device=dev), torch.randn(ntok, 192, device=dev).to(torch.bfloat16)
    add("k6_layernorm_fwd", tk(lambda: ops.layer_norm(xs, ln, "both")), ntok * 192 * (4 + 4 + 2), 12)
    # backward through the C-ABI directly (an autograd.grad call would time Python / autograd dispatch, not the kernel)
    from mobgt_b200 import _C as C_
    mean_, rstd_ = torch.empty(ntok, device=dev), torch.empty(ntok, device=dev)
    o32_, o16_ = torch.empty(ntok, 192, device=dev), torch.empty(ntok, 192, device=dev, dtype=torch.bfloat16)
    gam, bet = ln.weight.detach().float().contiguous(), ln.bias.detach().float().contiguous()
    C_.call("mobgt_layernorm_fwd", C_.ptr(xs), C_.ptr(gam), C_.ptr(bet), float(ln.eps), ntok, 192, C_.ptr(o32_), C_.ptr(o16_),
            C_.ptr(mean_), C_.ptr(rstd_), C_.stream_ptr())
    dx_, dg_, db_ = torch.empty_like(xs), torch.empty(192, device=dev), torch.empty(192, device=dev)
    wsb = int(C_.lib().mobgt_layernorm_bwd_workspace_bytes(192))
    ws_ = torch.empty(wsb, dtype=torch.uint8, device=dev)
    add("k6_layernorm_bwd", tk(lambda: C_.call("mobgt_layernorm_bwd", C_.ptr(dy32), C_.ptr(dy16), C_.ptr(xs), C_.ptr(gam), C_.ptr(mean_),
                                               C_.ptr(rstd_), ntok, 192, C_.ptr(dx_), C_.ptr(dg_), C_.ptr(db_), C_.ptr(ws_), wsb,
                                               C_.stream_ptr())),
        ntok * 192 * (4 + 2 + 4 + 4), 12)
    wide = torch.randn(ntok, 1024, device=dev).to(torch.bfloat16)
    wide2 = torch.randn(ntok, 1024, device=dev).to(torch.bfloat16)
    add("k6_gelu_bwd_colsum", tk(lambda: ops.gelu_bwd_colsum_raw(wide2, wide)), ntok * 1024 * (2 + 2 + 2), 6)
    del wide2
    add("k6_colsum_1024", tk(lambda: ops.colsum(wide)), ntok * 1024 * 2, 0)
    add("k6_colsum_192", tk(lambda: ops.colsum(dy16)), ntok * 192 * 2, 12)
    del wide
    # K10 — encoder GEMMs on tcgen05 with fused epilogues (SURVEY §8f #2): the three FFN shapes of a layer
    x16 = torch.randn(ntok, 192, device=dev).to(torch.bfloat16)
    w1_ = (torch.randn(1024, 192, device=dev) * 0.07).to(torch.bfloat16)
    w2_ = (torch.randn(192, 1024, device=dev) * 0.03).to(torch.bfloat16)
    b1_, b2_ = torch.randn(1024, device=dev) * 0.1, torch.randn(192, device=dev) * 0.1
    a16 = ops.gemm_bf16(x16, w1_, b1_, mode=1)
    w2t_ = w2_.t().contiguous()
    gflop = 2.0 * ntok * 192 * 1024
    add("k10_ffn1_gelu_fwd", tk(lambda: ops.gemm_bf16(x16, w1_, b1_, mode=1)), ntok * (192 + 1024) * 2 + 1024 * 192 * 2, 6, gflop)
    add("lib_ffn2_fwd", tk(lambda: F_.linear(a16, w2_, b2_.to(torch.bfloat16))), ntok * (192 + 1024) * 2 + 1024 * 192 * 2, 0, gflop)
    add("k10_ffn_bwd_dh", tk(lambda: ops.gemm_bf16(dy16, w2t_, b1_, mode=2, a2=x16, w2=w1_, want_colsum=True)),
        ntok * (192 + 192 + 1024) * 2 + 2 * 1024 * 192 * 2, 6, 2 * gflop)
    add("lib_ffn1_gemm_plus_gelu", tk(lambda: F_.gelu(F_.linear(x16, w1_, b1_.to(torch.bfloat16)))), ntok * (192 + 3 * 1024) * 2, 0, gflop)
    del x16, a16
    # K5 — the evaluation head (not part of the training step): c2 shape, and one GPU's shard of the c5 shape
    for name, Mh, Vh in (("k5_head_c2", 256, 60001),) + ((("k5_head_c5_shard", 4096, 125000),) if head_c5 else ()):
        g_ = torch.Generator(device=dev).manual_seed(5)
        z = torch.randn(Mh, 320, device=dev, generator=g_).to(torch.bfloat16)
        Wh = (torch.randn(Vh, 320, device=dev, generator=g_) * 0.02).to(torch.bfloat16)
        tgt = torch.randint(0, Vh, (Mh,), device=dev, generator=g_).int()
        st = ops.head_target_logit(z, Wh, None, tgt)
        add(name, tk(lambda: ops.head_topk_local(z, Wh, None, tgt, 10, st=st)), Vh * 320 * 2 + Mh * 320 * 2 + Mh * 10 * 8, 0,
            2.0 * Mh * 320 * Vh)
        del z, Wh
    del flush
    return rep


# ------------------------------------------------------------------------------------------------ ours
def _dist_setup():
    import torch.distributed as dist
    rank, world_size = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world_size > 1:
        dist.init_process_group("nccl", device_id=dev)
    return rank, world_size, local, dev


def _timed(fn, steps, dev, world_size, finalize=None):
    """K calls of fn bracketed by barrier + synchronize, timed with CUDA events on the current stream; max over ranks (ms)."""
    import torch.distributed as dist

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    if finalize is not None:
        finalize()
    b_.record()
    barrier()
    ms = torch.tensor([a.elapsed_time(b_)], device=dev)
    if world_size > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def run_ours(args):
    if args.workload == "c3-preprocess":
        return run_c3(args)
    if args.workload == "c5-eval":
        return run_c5(args)
    import torch.distributed as dist
    from mobgt_b200 import _C, collator, model as M
    from mobgt_b200.trainer import Trainer
    rank, world_size, local, dev = _dist_setup()
    _C.require_cuda()
    pk = peaks()
    cfg, ds, cap, n_fixed, nbatches = TRAIN_WORKLOADS[args.workload]
    world = make_world_for(args.workload)
    B = args.batch
    item_sets = [make_workload(args.workload, world, B, rank, batch_id=i) for i in range(nbatches)]
    torch.manual_seed(1)
    model = M.Graphormer(dataset_name=ds, world=world, **HP).to(dev).train()
    # the loop `python -m mobgt_b200.entry` runs: flat fp32 gradient buffer, CUDA-graph replay of repeated shapes, bucketed /
    # overlapped NCCL all-reduce, fused AdamW, PolynomialDecayLR
    tr = Trainer(model, dev, world_size, cuda_graph=args.cuda_graph, overlap=not args.no_overlap)
    latlon = torch.from_numpy(world.latlon).to(dev)
    ckw = dict(world=world, latlon_dev=latlon, multi_hop_max_dist=HP["multi_hop_max_dist"], rel_pos_max=1024, device=dev)
    bucket = nbatches > 1 and args.cuda_graph          # varying shapes: pad to size buckets so the captured graphs replay
    batches = [collator.collate_packed(its, max_node=512, bucket=bucket, **ckw) for its in item_sets]
    state = dict(i=0)

    def resident_step():
        b = batches[state["i"] % nbatches]
        state["i"] += 1
        state["loss"] = tr.train_step(b)

    for _ in range(max(args.warmup, 2 * nbatches)):       # every distinct shape is seen twice: repeated shapes get captured
        resident_step()
    n0, g0 = _C.launch_count(), tr.graph_steps
    sampler = ClockSampler(local) if rank == 0 else None
    ms = _timed(resident_step, args.steps, dev, world_size)
    if args.dump_outputs and rank == 0:        # now: the next step (a graph replay) overwrites the loss, the gradients, the weights
        outs = {"loss": state["loss"]}
        for name, p in model.named_parameters():
            outs["param." + name], outs["grad." + name] = p, p.grad
        dump_outputs(args.dump_outputs, outs)
    replays_value = tr.graph_steps - g0
    launches = (_C.launch_count() - n0) / args.steps + tr.graph_launches * replays_value / args.steps
    tokens = int(np.mean([int(b.tok_pos.numel()) for b in batches]))

    # ---- end to end: host items -> collate (pack + pinned H2D + K1 + poi_pos + sort plans) -> step -> loss on the host
    losses = []

    def endless():
        i = 0
        while True:
            yield item_sets[i % nbatches]
            i += 1

    # one-batch-ahead loader (the reference's DataLoader-worker role, data.py:255-267): numpy packing in worker processes, ONE
    # pinned buffer + ONE H2D copy per batch, collation kernels on a side stream gated behind the previous step
    side = not args.no_side_stream
    loader = collator.PackedLoader(endless(), num_workers=args.loader_workers, side_stream=side, bucket=bucket, **ckw)
    loss_pin = torch.empty(2, dtype=torch.float32).pin_memory()
    st = dict(pending=None, k=0, last=None)

    def e2e_flush():
        if st["pending"] is not None:
            ev, slot = st["pending"]
            ev.synchronize()
            losses.append(float(loss_pin[slot]))
            st["pending"] = None

    def e2e_step():
        b = loader.current()
        loss = tr.train_step(b)
        slot = st["k"] & 1
        loss_pin[slot:slot + 1].copy_(loss.detach().view(1), non_blocking=True)      # the step's result, read back every step
        ev = torch.cuda.Event()
        ev.record()
        loader.advance()
        e2e_flush()                       # the PREVIOUS step's loss (its event has long completed)
        st["pending"], st["k"], st["last"] = (ev, slot), st["k"] + 1, b

    # warm-up of the end-to-end path: at least max(6, W) steps, then in chunks of 5 until the loader pipeline (worker processes,
    # pinned staging buffers, the allocator's pool of collation buffers) has reached its steady state — on a freshly started
    # box the first tens of steps run 2-3 x slower (workers still starting / paging in); capped at 80 steps
    for _ in range(max(6, args.warmup)):
        e2e_step()
    e2e_flush()
    chunk_ms, stable = [], 0
    while len(chunk_ms) < 15 and stable < 2:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            e2e_step()
        e2e_flush()
        torch.cuda.synchronize()
        cur = (time.perf_counter() - t0) * 200.0
        stable = stable + 1 if (chunk_ms and abs(cur - min(chunk_ms)) <= 0.15 * min(chunk_ms)) else 0
        chunk_ms.append(cur)
    if rank == 0:
        print("[bench] e2e warm-up chunks (ms/step): " + " ".join(f"{x:.2f}" for x in chunk_ms), file=sys.stderr)
    e2e_steps = args.steps
    eg0, ee0 = tr.graph_steps, tr.eager_steps
    ms_e2e = _timed(e2e_step, e2e_steps, dev, world_size, finalize=e2e_flush)
    clocks = sampler.stop() if sampler else None
    h2d = int(st["last"].h2d_bytes)
    if rank == 0:
        graphs = B * world_size
        line = {"metric": "train_graphs_per_sec", "value": graphs * args.steps / (ms / 1e3), "unit": "graphs/s",
                "n_gpus": world_size, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": DATA_NOTE.get(cfg, "synthetic"),
                "config": {"workload": args.workload, "world": WORLD_NOTE[cfg], "hidden": 128, "layers": 6,
                           "heads": 8, "ffn": 1024, "multi_hop_max_dist": 20, "graphs_per_gpu": B,
                           "tokens_per_gpu": tokens, "distinct_batches": nbatches, "size_buckets": bool(bucket), "parallelism": f"dp{world_size}",
                           "cuda_graph": tr.graph_note, "graph_replays_of_timed_steps": f"{replays_value}/{args.steps}",
                           "e2e_graph_replays": f"{tr.graph_steps - eg0}/{e2e_steps}",
                           "allreduce": ("none" if world_size == 1 else
                                         "one NCCL all-reduce (AVG) of the flat fp32 gradient buffer after the graph replay; eager steps "
                                         "start the out_proj bucket during the backward"),
                           "e2e_collate_stream": "side" if side else "training",
                           "l2": "per-step working set (activations + bias planes, > 1 GB) exceeds the 126 MB L2"},
                "e2e": {"value": graphs * e2e_steps / (ms_e2e / 1e3), "unit": "graphs/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / e2e_steps},
                "gpu_launches": launches, "clocks": clocks, "final_loss": losses[-1] if losses else None}
        if world_size == 1 and not args.no_kernel_report:
            rep = kernel_report(model, batches[0], pk, head_c5=(cfg == "c2"))
            top = max(rep, key=lambda k: rep[k]["ms"] * rep[k]["launches_per_step"])
            r = rep[top]
            tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")      # dram bytes / launch from the committed ncu capture
            traffic = json.load(open(tp)).get(top) if (os.path.exists(tp) and args.workload == "c2-dense128") else None
            line["roofline"] = {"kernel": top, "bound": "hbm", "achieved": r["gbs"], "peak": pk["hbm"], "unit": "GB/s",
                                "frac": r["frac_hbm"], "traffic": traffic, "peak_source": pk["src"],
                                "share_of_step": r["ms"] * r["launches_per_step"] / (ms / args.steps)}
            line["kernels"] = {k: {kk: (round(vv, 4) if isinstance(vv, float) else vv) for kk, vv in v.items()} for k, v in rep.items()}
        if world_size == 1 and not args.no_cpu_baseline:
            r = cpu_reference_rate(args.workload, steps=4, warmup=2, full_batch=B)
            line["cpu_baseline"] = {"value": r["value"], "unit": "graphs/s", "cores": r["cores"], "kind": "port",
                                    "parts": {"algos": r["algos"], "collator+model": "port (oracle/model_oracle.py)"},
                                    "sample": _cpu_sample_text(r, 4, 2)}
        emit(line)
    if world_size > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ c5: sharded evaluation head
def run_c5(args):
    """BASELINE configs[4]: POI-logit head over a 1 M-POI vocabulary sharded by rows across the N GPUs; one step = 4 096 z rows
    through s_t (all-reduce MAX) -> fused GEMM + top-10 + rank count (K5) -> all-gather of the lists over NVLink -> all-reduce
    SUM of the counts -> merge -> Acc / NDCG / MRR sums."""
    import torch.distributed as dist
    from mobgt_b200 import _C, ops, parallel
    rank, world, local, dev = _dist_setup()
    _C.require_cuda()
    pk = peaks()
    V, M, k = args.vocab, args.rows, 10
    off, size = parallel.shard_vocab(V, rank, world)
    g = torch.Generator(device=dev).manual_seed(11)           # the same z / targets on every rank (replicated rows)
    z = torch.randn(M, 320, device=dev, generator=g).to(torch.bfloat16)
    target = torch.randint(1, V, (M,), device=dev, generator=g).int()
    gw = torch.Generator(device=dev).manual_seed(1000 + rank)  # this rank's vocabulary rows
    W = (torch.randn(size, 320, device=dev, generator=gw) * 0.02).to(torch.bfloat16)
    bias = torch.randn(size, device=dev, generator=gw) * 0.1
    res = {}

    def step():
        res["r"] = ops.head_topk_sharded(z, W, bias, target, k, off)

    for _ in range(args.warmup):
        step()
    n0 = _C.launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    ms = _timed(step, args.steps, dev, world)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res["r"])
    launches = (_C.launch_count() - n0) / args.steps
    # e2e: z rows and targets start in pinned HOST memory; top-k ids and ranks are read back to the host every step
    zh, th = z.cpu().pin_memory(), target.cpu().pin_memory()
    out_idx = torch.empty(M, k, dtype=torch.int32).pin_memory()
    out_rank = torch.empty(M, dtype=torch.int32).pin_memory()
    mets = {}

    def e2e_step():
        zd, td = zh.to(dev, non_blocking=True), th.to(dev, non_blocking=True)
        r = ops.head_topk_sharded(zd, W, bias, td, k, off)
        out_idx.copy_(r["idx"], non_blocking=True)
        out_rank.copy_(r["rank"], non_blocking=True)
        mets["r"], mets["t"] = r, td

    for _ in range(3):
        e2e_step()
    ms_e2e = _timed(e2e_step, args.steps, dev, world, finalize=torch.cuda.synchronize)
    clocks = sampler.stop() if sampler else None
    # dominant kernel alone (K5 on this rank's shard), L2 flushed between launches
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stl = ops.head_target_logit(z, W, bias, target, off)
    k5ms = time_kernel(lambda: ops.head_topk_local(z, W, bias, target, k, off, st=stl), flush, iters=8)
    del flush
    if rank == 0:
        m = ops.metrics_from_rank(mets["r"]["rank"], mets["t"].long(), ks=(1, 5, 10))
        fl = 2.0 * M * 320 * size
        line = {"metric": "eval_rows_per_sec", "value": M * args.steps / (ms / 1e3), "unit": "rows/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "c5-eval", "vocab": V, "rows_per_step": M, "k": k, "K": 320, "vocab_rows_per_gpu": size,
                           "parallelism": f"vocab-parallel x{world}",
                           "l2": "W shard (V/N x 320 bf16, >= 80 MB) streamed once per row tile; L2 flushed for the kernel-alone figure"},
                "e2e": {"value": M * args.steps / (ms_e2e / 1e3), "unit": "rows/s", "h2d_bytes_per_step": M * 320 * 2 + M * 4,
                        "d2h_bytes_per_step": M * k * 4 + M * 4, "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": launches, "clocks": clocks,
                "roofline": {"kernel": "k5_head_topk (this rank's shard)", "bound": "tensor", "achieved": fl / k5ms / 1e9, "peak": pk["tc"],
                             "unit": "TFLOP/s", "frac": fl / k5ms / 1e9 / pk["tc"], "traffic": None, "peak_source": pk["src"],
                             "ms": k5ms, "share_of_step": k5ms / (ms / args.steps)},
                "metrics": {kk: vv / M for kk, vv in m.items()}}
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = c5_cpu(V, 320, k)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def c5_cpu(V, K, k, seconds=15.0):
    """The reference's evaluation on the CPU (model_fqandtoyo.py:1396-1428 + get_acc :48-90 + MRR_metric :122-131): fp32 logits
    GEMM, topk(20) and a full descending argsort per row, on a bounded sample of rows against the full vocabulary."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(3)
    rows = 64
    z = torch.randn(rows, K, generator=g)
    W = torch.randn(V, K, generator=g) * 0.02
    b = torch.randn(V, generator=g) * 0.1
    t = torch.randint(1, V, (rows,), generator=g)
    done, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds or done == 0:
        logits = z @ W.t() + b
        logits.topk(20, 1)
        order = np.argsort(-logits.numpy(), axis=1)                  # MRR_metric's full sort (:128)
        (order == t.numpy()[:, None]).argmax(1)
        done += rows
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "rows/s", "cores": cores, "kind": "port",
            "sample": f"{done} rows x full {V}-POI vocabulary in {dt:.1f} s: fp32 GEMM + topk(20) + full argsort per row (get_acc / MRR_metric)"}


def run_c5_reference(args):
    r = c5_cpu(args.vocab, 320, 10, seconds=max(10.0, 2.0 * args.steps))
    emit({"metric": "eval_rows_per_sec", "value": r["value"], "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": 1e3 * args.rows / r["value"], "higher_is_better": True, "scaling": "strong",
          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
          "config": {"workload": "c5-eval", "vocab": args.vocab, "rows_per_step": args.rows, "k": 10, "K": 320},
          "cpu_baseline": r, "e2e": {"value": r["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


# ------------------------------------------------------------------------------------------------ c3: preprocessing
def _c3_items(args, rank, world_size):
    from mobgt_b200 import synth
    world = synth.make_world("c2", seed=1)
    per = args.graphs // world_size
    return synth.make_items(world, per, 512, seed=1, cfg_id=3, start=rank * per)


def _pack_planes(items):
    from mobgt_b200.algos import pack_graphs
    ns = np.array([len(np.asarray(it.x)) for it in items], np.int32)
    nn, sq, _ = pack_graphs(ns)
    feat = np.zeros(int(sq[-1]), np.uint8)
    for g, it in enumerate(items):
        ei = np.asarray(it.edge_index)
        feat[sq[g] + ei[0] * int(ns[g]) + ei[1]] = np.asarray(it.edge_attr).reshape(-1) + 2      # wrapper.py:49-53
    return nn, sq, feat


def run_c3(args):
    """BASELINE configs[2]: K1 over `--graphs` synthetic trajectory graphs <= 512 nodes (natural node-count law), sharded over
    the ranks with no collective.  One step = one pass over this rank's graphs in batches of 8 192."""
    import torch.distributed as dist
    from mobgt_b200 import _C
    from mobgt_b200.algos import apsp_edge_input_packed
    rank, world_size, local, dev = _dist_setup()
    _C.require_cuda()
    pk = peaks()
    items = _c3_items(args, rank, world_size)
    bs = 8192
    host = []
    for s0 in range(0, len(items), bs):
        nn, sq, feat = _pack_planes(items[s0:s0 + bs])
        host.append((nn, torch.from_numpy(nn).pin_memory(), torch.from_numpy(sq).pin_memory(), torch.from_numpy(feat).pin_memory()))
    resident = [(nn, a.to(dev), b.to(dev), c.to(dev)) for nn, a, b, c in host]
    cells = sum(int(b[-1]) for _, _, b, _ in host)
    ops_minplus = float(sum(2.0 * (nn.astype(np.float64) ** 3).sum() for nn, _, _, _ in host))
    keep = {}

    def step_resident():
        for nn, nd, sd, fd in resident:
            keep["o"] = apsp_edge_input_packed(fd, nd, sd, nn, 20, 1)

    def step_e2e():
        for nn, nd, sd, fd in host:
            o = apsp_edge_input_packed(fd.to(dev, non_blocking=True), nd.to(dev, non_blocking=True), sd.to(dev, non_blocking=True), nn, 20, 1)
            keep["md"] = o["maxdist"].to("cpu", non_blocking=True)       # the per-graph max_dist (wrapper.py:58) is read back

    for _ in range(min(args.warmup, 3)):
        step_resident()
    n0 = _C.launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    ms = _timed(step_resident, args.steps, dev, world_size)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, keep["o"])
    launches = (_C.launch_count() - n0) / args.steps
    step_e2e()
    ms_e2e = _timed(step_e2e, args.steps, dev, world_size, finalize=torch.cuda.synchronize)
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        G = len(items) * world_size
        alg = cells * 23.0
        int_peak = 148 * 4 * 16 * 2 * 1.965e9 / 1e12      # u16x2 min-plus per clk: 148 SMs x 4 SMSPs x 16 lanes x 2 halves, T op/s
        line = {"metric": "preprocess_graphs_per_sec", "value": G * args.steps / (ms / 1e3), "unit": "graphs/s", "n_gpus": world_size,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "u16", "data": "synthetic",
                "config": {"workload": "c3-preprocess", "graphs": G, "node_cap": 512, "law": "Gowalla-Nevada node-count histogram",
                           "hops": 20, "batch": bs, "l2": "each pass streams new graphs; outputs (23 B/cell) written once"},
                "e2e": {"value": G * args.steps / (ms_e2e / 1e3), "unit": "graphs/s", "h2d_bytes_per_step": cells + 12 * len(items),
                        "d2h_bytes_per_step": 4 * len(items), "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": launches, "clocks": clocks,
                "roofline": {"kernel": "k1_apsp_kernel", "bound": "hbm", "achieved": alg / (ms / args.steps) / 1e6, "peak": pk["hbm"],
                             "unit": "GB/s", "frac": alg / (ms / args.steps) / 1e6 / pk["hbm"], "traffic": None, "peak_source": pk["src"],
                             "int_alu": {"achieved_T_minplus_per_s": ops_minplus / (ms / args.steps) / 1e9,
                                         "peak_T_minplus_per_s": int_peak, "frac": ops_minplus / (ms / args.steps) / 1e9 / int_peak}}}
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = c3_cpu(items, seconds=15.0)
        emit(line)
    if world_size > 1:
        dist.destroy_process_group()


def _c3_worker(i):
    from helpers import run_algos
    it = _PRE["items"][i]
    ei = np.asarray(it.edge_index)
    run_algos(_PRE["algos"], len(np.asarray(it.x)), ei[0], ei[1], np.asarray(it.edge_attr).reshape(-1))     # wrapper.py:55-60
    return 1


def c3_cpu(items, seconds=15.0):
    """algos.pyx driven like wrapper.py:55-60 (FW -> max -> gen_edge_input(max_dist) -> slice) in min(8, cores) worker
    processes (README.md:62), on a bounded prefix of the same graphs."""
    import multiprocessing as mp
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import algos_oracle
    import build_ref
    ref = build_ref.load()
    cores = os.cpu_count() or 1
    workers = min(8, cores)
    _PRE.update(items=items, algos=ref if ref is not None else algos_oracle)
    pool = mp.get_context("fork").Pool(workers, initializer=_pre_init)
    done, t0 = 0, time.perf_counter()
    try:
        chunk = 256
        while done < len(items) and time.perf_counter() - t0 < seconds:
            done += sum(pool.map(_c3_worker, range(done, min(len(items), done + chunk)), chunksize=8))
    finally:
        pool.terminate()
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "graphs/s", "cores": workers, "kind": "reference" if ref is not None else "port",
            "sample": f"the first {done} graphs of the same set in {dt:.1f} s: {'compiled algos.pyx (oracle/_ref)' if ref is not None else 'C port (oracle/algos_oracle.c)'} "
                      f"floyd_warshall + gen_edge_input(max_dist) as wrapper.py:55-60, {workers} worker processes"}


def run_c3_reference(args):
    items = _c3_items(args, 0, 1)
    r = c3_cpu(items, seconds=max(15.0, 3.0 * args.steps))
    emit({"metric": "preprocess_graphs_per_sec", "value": r["value"], "unit": "graphs/s", "n_gpus": args.gpus, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": 1e3 * len(items) / r["value"], "higher_is_better": True, "scaling": "strong",
          "vs_baseline": None, "dtype": "i64", "data": "synthetic", "impl": "reference",
          "config": {"workload": "c3-preprocess", "graphs": len(items), "node_cap": 512, "hops": 20},
          "cpu_baseline": r, "e2e": {"value": r["value"], "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2-dense128",
                    choices=["c2-dense128", "c2-natural", "c4-gowalla256", "c4-dense256", "c4-gowalla-real", "c5-eval", "c3-preprocess"])
    ap.add_argument("--vocab", type=int, default=1_000_000, help="c5-eval: POI vocabulary (sharded across the GPUs)")
    ap.add_argument("--rows", type=int, default=4096, help="c5-eval: z rows per step")
    ap.add_argument("--graphs", type=int, default=100_000, help="c3-preprocess: graphs per pass")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1: one flat all-reduce after the backward (no early bucket)")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--loader-workers", type=int, default=2, help="DataLoader worker processes packing raw items (e2e path)")
    ap.add_argument("--no-side-stream", action="store_true", help="e2e: collate on the training stream (no overlap)")
    ap.add_argument("--no-cuda-graph", dest="cuda_graph", action="store_false", help="run every step eagerly")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-report", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(3, args.warmup)
    # stdout carries exactly ONE JSON line: everything libraries print to fd 1 meanwhile (the NCCL version banner, ...) goes to
    # stderr; the line is written to the saved descriptor at the end
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
