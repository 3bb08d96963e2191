"""`entry.py` of the reference (graphormer/entry.py:48-165) with the same flag surface, driving the B200-native hot path.

    python -m mobgt_b200.entry --dataset_name toyotagraph --gpus 1 --batch_size 256 --hidden_dim 128 --num_heads 8 \
        --n_layers 6 --ffn_dim 1024 --dropout_rate 0.1 --peak_lr 2e-4 --edge_type multi_hop --multi_hop_max_dist 20 \
        --warmup_updates 40000 --tot_updates 400000 --seed 1 --max_epochs 1 --default_root_dir exps/toyota
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 -m mobgt_b200.entry --accelerator ddp ...

Flag groups (names and defaults as in the reference):
  * model:      Graphormer.add_model_specific_args                      (model_fqandtoyo.py:1619-1641)
  * datamodule: --dataset_name --num_workers --batch_size --seed --multi_hop_max_dist --rel_pos_max   (data.py:197-207)
  * trainer:    the pytorch_lightning.Trainer flags the README uses      (README.md:62): --gpus --accelerator --precision
                --max_epochs --max_steps --check_val_every_n_epoch --default_root_dir --resume_from_checkpoint
The Lightning runtime itself is out of scope (SURVEY.md §2 #9): `mobgt_b200.trainer.Trainer` replaces it — the SAME class
`bench.py` times: data-parallel over trajectory graphs (every rank gets the same number of graphs, like DistributedSampler),
one-batch-ahead collation (`collator.PackedLoader`, `--num_workers` packing processes), CUDA-graph replay of fixed-shape
steps, one all-reduce of the flat fp32 gradient buffer per step (its out_proj bucket overlapped with the backward),
`last.ckpt` auto-resume (entry.py:135-137), and at test time the fused K5 head + the reference's three metric lines
(model_fqandtoyo.py:1593-1595) over the metric sums of ALL ranks.

The reference reads ../dataset/<name>/raw/*; those blobs are not shipped (SURVEY.md §0.5), so the data here is the
seeded synthetic world of mobgt_b200.synth (`--synthetic` picks the BASELINE.json shape, `--train_graphs` the split size).
"""
import argparse
import os
import time

import numpy as np
import torch

DATASET_DEFAULT_SHAPE = {"foursquaregraph": "c1", "toyotagraph": "c2", "gowalla_nevda": "c4", "gowalla_7day": "c4"}
COLLATORS = {"foursquaregraph": "collator_foursquare", "toyotagraph": "collator_toyota", "gowalla_nevda": "collator_gowalla",
             "gowalla_7day": "collator_gowalla"}


def build_parser():
    from .model import Graphormer
    parser = argparse.ArgumentParser(description="MobGT (B200-native hot path)")
    t = parser.add_argument_group("pl.Trainer")                         # entry.py:53
    t.add_argument("--gpus", type=int, default=1)
    t.add_argument("--accelerator", type=str, default=None)             # "ddp" -> one rank per GPU (launched by torchrun)
    t.add_argument("--precision", type=int, default=16, choices=(16, 32))   # 16: bf16 GEMMs / attention (the reference: fp16 AMP); 32: fp32 path
    t.add_argument("--max_epochs", type=int, default=1)
    t.add_argument("--max_steps", type=int, default=None)               # overwritten from tot_updates (entry.py:57)
    t.add_argument("--check_val_every_n_epoch", type=int, default=1)
    t.add_argument("--default_root_dir", type=str, default="exps/mobgt")
    t.add_argument("--resume_from_checkpoint", type=str, default=None)
    t.add_argument("--progress_bar_refresh_rate", type=int, default=50)
    Graphormer.add_model_specific_args(parser)                          # entry.py:54
    d = parser.add_argument_group("GraphDataModule")                    # entry.py:55 / data.py:197-207
    d.add_argument("--dataset_name", type=str, default="toyotagraph")
    d.add_argument("--num_workers", type=int, default=0)
    d.add_argument("--batch_size", type=int, default=256)
    d.add_argument("--seed", type=int, default=1)
    d.add_argument("--multi_hop_max_dist", type=int, default=5)
    d.add_argument("--rel_pos_max", type=int, default=1024)
    d.add_argument("--max_node", type=int, default=512,
                   help="largest trajectory graph (nodes) a batch takes; larger ones are left out of every epoch (collator.py:313). "
                        "Up to 512 by default; 513..1024 turns on the collator's large_graphs mode (the reference: 30000, data.py)")
    s = parser.add_argument_group("synthetic data (stand-in for ../dataset/<name>) and run options of this implementation")
    s.add_argument("--synthetic", type=str, default=None, help="c1|c2|c4|tiny (default: by dataset_name)")
    s.add_argument("--train_graphs", type=int, default=2048)
    s.add_argument("--test_graphs", type=int, default=512)
    s.add_argument("--n_fixed", type=int, default=None, help="every synthetic graph gets exactly this many nodes")
    s.add_argument("--data_root", type=str, default=None,
                   help="a dataset directory in the reference's on-disk format (<root>/raw/{train,test}.pickle, *_idx.pkl, "
                        "Graph_{poi,dist,cat}.csv: ../dataset/<name> of the reference) instead of synthetic data")
    s.add_argument("--data_npz", type=str, default=None,
                   help="the same data set in the compact form of mobgt_b200.owndata.pack_dataset (e.g. the real Gowalla-Nevada "
                        "fixture tests/golden/gowalla_nevda_real.npz)")
    s.add_argument("--limit_train_steps", type=int, default=None, help="stop after this many optimizer steps (smoke runs)")
    s.add_argument("--no_cuda_graph", action="store_true", help="never capture the step in a CUDA graph")
    s.add_argument("--eval_vocab_parallel", action="store_true",
                   help="evaluation head with out_proj sharded by vocabulary rows across the ranks (SURVEY.md §8e)")
    return parser


def parse_args(argv=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    if not 1 <= args.max_node <= 1024:
        parser.error(f"--max_node {args.max_node}: the model's kernels take graphs of 1 to 1024 nodes")
    args.max_steps = args.tot_updates + 1                               # entry.py:57
    return args


def _ckpt_dir(args):
    return os.path.join(args.default_root_dir, "lightning_logs", "checkpoints")     # entry.py:123


def cli_main(argv=None):
    """-> dict(loss=last training loss | None, metrics=last evaluation | None, steps=optimizer steps run)"""
    import torch.distributed as dist
    from . import _C, collator, parallel, synth
    from .model import Graphormer
    from .trainer import Trainer
    args = parse_args(argv)
    rank, world_size = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    _C.require_cuda()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    own_pg = False
    if world_size > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
        own_pg = True
    if rank == 0 and not args.test and not args.validate:
        print(args)
    torch.manual_seed(args.seed)                                        # pl.seed_everything (entry.py:60)
    np.random.seed(args.seed)

    if args.data_root or args.data_npz:                                 # the reference's data set (owndata.py, model ctor tables)
        from . import owndata
        if args.data_npz:
            world, splits = owndata.unpack_dataset(np.load(args.data_npz))
            world.dataset_name = args.dataset_name
            train, test = splits["train"], splits["test"]
        else:
            raw = os.path.join(args.data_root, "raw")
            world = owndata.load_world(raw, args.dataset_name)
            train, test = owndata.load_items(raw, "train"), owndata.load_items(raw, "test")
        if rank == 0:
            print(f"data set: {len(train)} train / {len(test)} test trajectories, {world.P} POIs, {world.C} categories")
    else:
        shape = args.synthetic or DATASET_DEFAULT_SHAPE.get(args.dataset_name, "c2")
        world = synth.make_world(shape, seed=args.seed, dataset_name=args.dataset_name)
        cap = synth.CONFIGS[shape]["cap"]
        train = synth.make_items(world, args.train_graphs, cap, seed=args.seed, cfg_id=11, n_fixed=args.n_fixed)
        test = synth.make_items(world, args.test_graphs, cap, seed=args.seed, cfg_id=12, n_fixed=args.n_fixed)
    latlon = torch.from_numpy(world.latlon).to(dev)
    ckw = dict(world=world, latlon_dev=latlon, multi_hop_max_dist=args.multi_hop_max_dist, rel_pos_max=args.rel_pos_max, device=dev)

    def item_batches(items, shuffle, epoch, pad):
        """This rank's share of the epoch as lists of raw items (DistributedSampler semantics, parallel.shard_graphs)."""
        order = np.arange(len(items))
        if shuffle:
            np.random.default_rng([args.seed, epoch]).shuffle(order)
        mine = parallel.shard_graphs(len(items), rank, world_size, order=order.tolist(), pad=pad)
        for i in range(0, len(mine), args.batch_size):
            yield [items[j] for j in mine[i:i + args.batch_size]]

    def loader(items, shuffle, epoch, pad):
        # one batch ahead: host packing in --num_workers processes, H2D + K1 + poi_pos + sort plans on a side stream; training
        # batches are padded to size buckets so that the captured CUDA graphs replay across batches of different graphs
        return collator.PackedLoader(item_batches(items, shuffle, epoch, pad), num_workers=args.num_workers, max_node=args.max_node,
                                     bucket=shuffle and not args.no_cuda_graph and args.precision == 16,
                                     large_graphs=args.max_node > _C.MAX_NODES, **ckw)

    model = Graphormer(
        n_layers=args.n_layers, num_heads=args.num_heads, hidden_dim=args.hidden_dim,
        attention_dropout_rate=args.attention_dropout_rate, dropout_rate=args.dropout_rate,
        intput_dropout_rate=args.intput_dropout_rate, weight_decay=args.weight_decay, ffn_dim=args.ffn_dim,
        dataset_name=args.dataset_name, warmup_updates=args.warmup_updates, tot_updates=args.tot_updates, peak_lr=args.peak_lr,
        end_lr=args.end_lr, edge_type=args.edge_type, multi_hop_max_dist=args.multi_hop_max_dist, flag=args.flag,
        flag_m=args.flag_m, flag_step_size=args.flag_step_size, world=world, precision=args.precision).to(dev)
    if args.checkpoint_path != "":                                      # entry.py:71-93 (strict=False)
        sd = torch.load(args.checkpoint_path, map_location=dev)
        model.load_state_dict(sd.get("state_dict", sd), strict=False)
    if rank == 0:
        print("total params:", sum(p.numel() for p in model.parameters()))

    # the fp32 mode is the full-precision / verification mode: it runs eagerly (CUDA-graph capture is exercised, and measured,
    # on the bf16 path only)
    use_graph = not args.no_cuda_graph and args.precision == 16
    tr = Trainer(model, dev, world_size, cuda_graph=use_graph)
    ckdir = _ckpt_dir(args)
    last = os.path.join(ckdir, "last.ckpt")
    epoch0 = 0
    resume = args.resume_from_checkpoint
    if not args.test and not args.validate and os.path.exists(last):    # entry.py:135-137
        resume = last
    if resume:
        ck = torch.load(resume, map_location=dev)
        tr.load_state_dict(ck, with_optimizer=not (args.test or args.validate))
        epoch0 = 0 if (args.test or args.validate) else int(ck.get("epoch", 0))
        if rank == 0:
            print("args.resume_from_checkpoint", resume)

    def evaluate(items):
        return tr.evaluate(loader(items, False, 0, pad=False), vocab_parallel=args.eval_vocab_parallel)

    result = dict(loss=None, metrics=None, steps=0)
    if args.test or args.validate:
        result["metrics"] = evaluate(test)                              # entry.py:146-154
        if rank == 0:
            print(result["metrics"])
    else:
        model.train()
        t0 = time.time()
        limit = args.max_steps if args.limit_train_steps is None else min(args.max_steps, tr.step_count + args.limit_train_steps)
        loss = None
        result["train_graphs"] = 0                                      # graphs trained on, summed over the epochs run
        for epoch in range(epoch0, args.max_epochs):
            ld = loader(train, True, epoch, pad=True)
            b = ld.current()
            while b is not None and tr.step_count < limit:
                loss = tr.train_step(b)
                result["train_graphs"] += int(b.B)
                ld.advance()                                            # collate the next batch under this step's kernels
                b = ld.current()
                if rank == 0 and tr.step_count % max(1, args.progress_bar_refresh_rate) == 0:
                    print(f"epoch {epoch} step {tr.step_count} train_loss {loss.item():.5f} lr {tr.sched.get_last_lr()[0]:.3e} "
                          f"({time.time() - t0:.1f}s)")
            if (epoch + 1) % args.check_val_every_n_epoch == 0:
                result["metrics"] = evaluate(test)
            if rank == 0:
                os.makedirs(ckdir, exist_ok=True)
                ck = tr.state_dict()
                ck.update(epoch=epoch + 1, hyper_parameters=vars(args))
                torch.save(ck, last)
            if tr.step_count >= limit:
                break
        result["loss"] = float(loss) if loss is not None else None
        result["steps"] = tr.step_count
        result["graph_steps"] = tr.graph_steps
        if rank == 0:
            print(f"trained {tr.step_count} steps: {tr.graph_steps} CUDA-graph replays, {tr.eager_steps} eager ({tr.graph_note})")
    if own_pg:
        dist.destroy_process_group()
    return result


if __name__ == "__main__":
    cli_main()
