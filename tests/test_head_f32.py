"""K5 in fp32 mode (csrc/k5_head_f32.cu, `mobgt_head_topk_f32`): the evaluation head of `--precision 32` computes its logits
in IEEE fp32 (one fmaf chain per logit, k ascending, then + bias) and ranks them with the same top-k / rank contract as the
bf16 head.

CPU: the C ABI rejects bad arguments before any launch.
GPU, kernel level: dumped logits within the fp32 error bound of float64; top-k, ids and ranks exactly consistent with the
kernel's own logits; ranks against float64 off by at most the logits inside the error band; exact ties (duplicated W rows)
go to the lower index; bitwise reproducibility across runs, split counts and vocabulary shards.
GPU, model level: `Graphormer(precision=32)` evaluation (test_step / test_epoch_end, `entry --precision 32 --test`) ranks
like the oracle's float64 logits; precision 16 keeps the bf16 head."""
import gc
import os
import sys

import numpy as np
import pytest
import torch

import model_oracle as mo

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NPZ = os.path.join(HERE, "golden", "gowalla_nevda_real.npz")
EPS = 2.0 ** -24


@pytest.fixture(autouse=True)
def _free_after_test():
    """Models, loaders and their CUDA events are released when each test ends, not by a garbage-collector pass that could fall
    inside a later test's CUDA-graph capture."""
    yield
    gc.collect()


# ------------------------------------------------------------------------------------------------------------- CPU: ABI
def _call(L, z=16, W=16, bias=None, target=16, M=8, V=100, K=320, off=0, k=10, nsplit=8, mode=1, st=16, outs=16):
    return L.mobgt_head_topk_f32(z, W, bias, target, M, V, K, off, k, nsplit, mode, st, outs, outs, outs, outs, None, None, None)


def test_abi_rejects_bad_arguments(lib_built):
    """Null pointers, K outside {4, 8, ..., 320}, k outside [1, 32], a bad split count and misaligned z / W: an error status
    and a message naming the limit, before anything touches the (here fake, host) pointers."""
    from mobgt_b200 import _C
    L = _C.lib()
    assert _call(L, z=None) == -6 and "null" in _C.last_error()
    assert _call(L, W=None) == -6
    assert _call(L, target=None) == -6
    assert _call(L, st=None) == -6
    assert _call(L, outs=None) == -6 and "null output" in _C.last_error()
    for K in (0, 2, 6, 322, 324, 640):
        assert _call(L, K=K) == -1, K
        assert "multiple of 4 in [4, 320]" in _C.last_error()
    for k in (0, 33, -1):
        assert _call(L, k=k) == -1, k
        assert "[1, 32]" in _C.last_error()
    for ns in (0, 2, 6, 164):
        assert _call(L, nsplit=ns) == -1, ns
        assert "multiple of 4 in [4, 160]" in _C.last_error()
    assert _call(L, mode=2) == -1
    assert _call(L, z=16 + 4) == -1 and "16-byte aligned" in _C.last_error()
    assert _call(L, W=16 + 8) == -1 and "16-byte aligned" in _C.last_error()
    assert _call(L, M=-1) == -1
    # the limits are inclusive; M = 0 returns before any launch
    assert _call(L, M=0, K=4, k=1, nsplit=4) == 0
    assert _call(L, M=0, K=320, k=32, nsplit=160) == 0


def test_split_rule_fits_the_merge():
    from mobgt_b200 import ops
    for M in (1, 24, 64, 65, 256, 1000, 4096):
        for V in (1, 100, 129, 3680, 60001, 125000):
            ns = ops.head_split(M, V, torch.float32)
            assert ns % 4 == 0 and 4 <= ns <= 160, (M, V, ns)
            assert ns // 4 <= (V + 127) // 128
    assert ops.head_split(256, 60001) == ops.head_split(256, 60001, torch.bfloat16)


# ------------------------------------------------------------------------------------------------------- GPU: kernel
def _case(M, V, K, seed=0, neg=0):
    g = torch.Generator().manual_seed(seed)
    z = torch.nn.functional.elu(torch.nn.functional.layer_norm(torch.randn(M, K, generator=g), (K,)))
    W = (torch.rand(V, K, generator=g) * 2 - 1) / K ** 0.5                 # nn.Linear's default initialisation
    bias = (torch.rand(V, generator=g) * 2 - 1) / K ** 0.5
    target = torch.randint(0, V, (M,), generator=g).int()
    if neg:
        target[torch.randperm(M, generator=g)[:neg]] = -1
    return z, W, bias, target


def _bound(z, W, bias):
    """Per-logit error bound of a K-step fmaf chain + one add, in float64: 1.01 (K+1) 2^-24 (sum |z_k w_k| + |b|)."""
    K = z.shape[1]
    a = z.double().abs() @ W.double().abs().t()
    if bias is not None:
        a = a + bias.double().abs().view(1, -1)
    return 1.01 * (K + 1) * EPS * a


def _ref64(z, W, bias):
    r = z.double() @ W.double().t()
    return r + bias.double().view(1, -1) if bias is not None else r


def _own_rank(L, st, t):
    """rank = #(s > s_t) + #(s == s_t and j < t) over the kernel's own logits (target < 0: st = -inf, t = -1)."""
    j = torch.arange(L.shape[1]).view(1, -1)
    return (L > st.view(-1, 1)).sum(1) + ((L == st.view(-1, 1)) & (j < t.long().view(-1, 1))).sum(1)


def _run(z, W, bias, target, k, **kw):
    from mobgt_b200 import ops
    out = ops.head_topk_local(z.cuda(), W.cuda(), None if bias is None else bias.cuda(), target.cuda(), k, **kw)
    torch.cuda.synchronize()
    return {n: (v.cpu() if torch.is_tensor(v) else v) for n, v in out.items()}


KERNEL_CASES = [
    # M, V, K, k, targets < 0, bias
    (256, 60001, 320, 20, 3, True),       # the c2 evaluation shape
    (100, 3001, 192, 10, 0, True),        # K of hidden_dim 64
    (65, 129, 320, 1, 5, True),           # one row past a 64-row tile, one column past a 128-column tile
    (7, 130, 192, 32, 1, False),
    (130, 5003, 320, 32, 0, True),
    (200, 20011, 192, 20, 2, False),
    (3, 1000, 4, 10, 0, True),            # K = 4: a single partial K chunk
    (70, 777, 36, 20, 0, True),           # K = 36: one full and one partial K chunk
]


@pytest.mark.gpu
@pytest.mark.parametrize("M,V,K,k,neg,with_bias", KERNEL_CASES)
def test_head_f32_logits_topk_and_rank(lib_built, M, V, K, k, neg, with_bias):
    z, W, bias, target = _case(M, V, K, seed=M + V + K, neg=neg)
    if not with_bias:
        bias = None
    out = _run(z, W, bias, target, k, dump_logits=True)
    L = out["logits"]
    ref = _ref64(z, W, bias)
    bnd = _bound(z, W, bias)
    # (1) fp32 arithmetic: every logit within the bound of the float64 value
    assert ((L.double() - ref).abs() <= bnd).all()
    # (2) s_t is the dumped logit of the target, bit for bit (mode 0 runs the same chain); -inf for target < 0
    live = target >= 0
    tl = target.long().clamp(min=0)
    assert torch.equal(out["st"][live], L.gather(1, tl.view(-1, 1)).view(-1)[live])
    assert torch.isneginf(out["st"][~live]).all()
    # (3) top-k values / ids and ranks exactly those of the kernel's own logits (ties -> lower index)
    order = torch.argsort(-L, dim=1, stable=True)[:, :k]
    assert torch.equal(out["idx"].long(), order)
    assert torch.equal(out["val"], L.gather(1, order))
    assert torch.equal(out["cnt"].long(), _own_rank(L, out["st"], target))
    # (4) against float64: a rank moves only by the logits inside the error band around s_t
    ref_t = ref.gather(1, tl.view(-1, 1))
    band = bnd + bnd.gather(1, tl.view(-1, 1))
    j = torch.arange(V).view(1, -1)
    rank64 = (ref > ref_t).sum(1) + ((ref == ref_t) & (j < tl.view(-1, 1))).sum(1)
    inside = (((ref - ref_t).abs() <= band) & (j != tl.view(-1, 1))).sum(1)
    assert ((out["cnt"].long() - rank64).abs() <= inside)[live].all()


@pytest.mark.gpu
def test_head_f32_ties_go_to_the_lower_index(lib_built):
    """Duplicated W rows (and biases) give bitwise-equal logits: top-k and the rank follow the lower-index rule, including
    rows that duplicate the target's own row before and after it."""
    M, V, K, k = 96, 3000, 320, 32
    z, W, bias, target = _case(M, V, K, seed=11)
    g = torch.Generator().manual_seed(12)
    src = torch.randint(0, 40, (V,), generator=g)
    dup = torch.rand(V, generator=g) < 0.7
    dup[:40] = False                                                                   # the source rows stay themselves
    W[dup] = W[src[dup]]
    bias[dup] = bias[src[dup]]
    target[: M // 2] = torch.randint(0, 40, (M // 2,), generator=g).int()           # targets with equal rows on both sides
    target[M // 2:] = torch.randint(2000, V, (M - M // 2,), generator=g).int()
    W[target[M // 2:].long()] = W[5].clone()
    bias[target[M // 2:].long()] = bias[5].clone()
    out = _run(z, W, bias, target, k, dump_logits=True)
    L = out["logits"]
    st = L.gather(1, target.long().view(-1, 1))
    j = torch.arange(V).view(1, -1)
    assert (((L == st) & (j < target.long().view(-1, 1))).sum(1) > 0).float().mean() >= 0.4    # ties before the target
    assert (((L == st) & (j > target.long().view(-1, 1))).sum(1) > 0).float().mean() >= 0.4    # and after it
    order = torch.argsort(-L, dim=1, stable=True)[:, :k]
    assert torch.equal(out["idx"].long(), order)
    assert torch.equal(out["cnt"].long(), _own_rank(L, st.view(-1), target))


@pytest.mark.gpu
def test_head_f32_is_bitwise_reproducible_across_runs_and_splits(lib_built):
    from mobgt_b200 import ops
    M, V, K, k = 300, 20011, 320, 20
    z, W, bias, target = _case(M, V, K, seed=5, neg=2)
    runs = [_run(z, W, bias, target, k, dump_logits=True) for _ in range(2)]
    runs += [_run(z, W, bias, target, k, dump_logits=True, nsplit=ns) for ns in (4, 12, 160)]
    assert ops.head_split(M, V, torch.float32) not in (4, 12, 160)
    for r in runs[1:]:
        for n in ("val", "idx", "cnt", "st", "logits"):
            assert torch.equal(r[n].view(torch.int32) if r[n].dtype == torch.float32 else r[n],
                               runs[0][n].view(torch.int32) if runs[0][n].dtype == torch.float32 else runs[0][n]), n


@pytest.mark.gpu
def test_head_f32_vocab_shards_merge_to_the_unsharded_result(lib_built):
    """Two vocabulary shards through the exchange steps of parallel.sharded_head_topk (s_t: MAX, lists: merge, counts: SUM),
    on one GPU: bitwise the unsharded result.  parallel.vocab_parallel_eval_head on one rank is the unsharded result too."""
    from mobgt_b200 import ops, parallel
    M, V, K, k = 200, 20001, 192, 10
    z, W, bias, target = _case(M, V, K, seed=3, neg=1)
    zc, Wc, bc, tc = z.cuda(), W.cuda(), bias.cuda(), target.cuda()
    full = ops.head_topk_local(zc, Wc, bc, tc, k)
    cut = 9000
    shards = [(0, Wc[:cut].contiguous(), bc[:cut].contiguous()), (cut, Wc[cut:].contiguous(), bc[cut:].contiguous())]
    st = torch.stack([ops.head_target_logit(zc, w, b, tc, off) for off, w, b in shards]).max(0).values
    assert torch.equal(st, full["st"])
    loc = [ops.head_topk_local(zc, w, b, tc, k, off, st=st) for off, w, b in shards]
    val, idx = ops.topk_merge_lists(torch.stack([l["val"] for l in loc], 1), torch.stack([l["idx"] for l in loc], 1))
    assert torch.equal(idx, full["idx"]) and torch.equal(val.view(torch.int32), full["val"].view(torch.int32))
    assert torch.equal(loc[0]["cnt"] + loc[1]["cnt"], full["cnt"])
    one = parallel.vocab_parallel_eval_head(ops, zc, Wc, bc, tc, k)
    assert torch.equal(one["idx"], full["idx"]) and torch.equal(one["rank"], full["cnt"])


# -------------------------------------------------------------------------------------------------------- GPU: model
def _oracle64_z(om, ob):
    """z (the [B, 2 hidden + 64] input of out_proj) from the oracle run in float64 on the same batch."""
    import copy
    om64 = copy.deepcopy(om).double()
    om64.D_A, om64.C_A = om64.D_A.double(), om64.C_A.double()
    ob64 = copy.copy(ob)
    for n, v in list(vars(ob).items()):
        if torch.is_tensor(v) and v.dtype == torch.float32 and n != "time_normal":
            setattr(ob64, n, v.double())
    with torch.no_grad():
        _, inner = om64(ob64, return_internals=True)
    return inner["z"], om64.out_proj.weight.detach(), om64.out_proj.bias.detach()


def _check_model_eval_vs_float64(pm, om, pb, ob, y_true):
    """test_step's top-20 ids / ranks and test_epoch_end's sums against the oracle's float64 logits.  Our logits (the fp32
    head's own, dumped for the same z) sit within 1e-5 x max |logit| of float64, the fp32 mode's contract; a logit's band is its
    actual distance d_j from float64 (encoder and head rounding together), and rows where another logit lies within
    |d_j| + |d_t| of the target's, the only rows whose rank may move, are excluded."""
    from mobgt_b200 import ops
    with torch.no_grad():
        out = pm.test_step(pb)
        z32, _ = pm.features(pb)
    y = y_true.cpu().long().view(-1)
    W32, b32 = pm.out_proj.weight.detach(), pm.out_proj.bias.detach()
    L32 = ops.head_topk_local(z32.detach().float().contiguous(), W32, b32, y_true.int().contiguous(), 20, dump_logits=True)["logits"]
    z64, W64, b64 = _oracle64_z(om, ob)
    s64 = z64 @ W64.t() + b64                          # raw logits: log_softmax (toyotagraph) is monotone per row
    d = (L32.cpu().double() - s64).abs()
    assert d.max().item() <= 1e-5 * s64.abs().max().item(), d.max().item()
    s_t = s64.gather(1, y.view(-1, 1))
    j = torch.arange(s64.shape[1]).view(1, -1)
    near = (((s64 - s_t).abs() <= d + d.gather(1, y.view(-1, 1))) & (j != y.view(-1, 1))).any(1)
    assert near.float().mean() <= 0.25, (int(near.sum()), len(y))
    band = 2 * d.max(1).values
    ok = ~near
    rank64 = (s64 > s_t).sum(1)
    assert torch.equal(out["rank"].cpu().long()[ok], rank64[ok])
    tv, ti = s64.topk(21, dim=1)
    decisive = ((tv[:, :-1] - tv[:, 1:]) > band.view(-1, 1)).all(1)
    assert decisive.float().mean() >= 0.5
    assert torch.equal(out["idx"].cpu().long()[decisive], ti[:, :20][decisive])
    sub = {"rank": out["rank"][ok.to(out["rank"].device)], "y_true": out["y_true"][ok.to(out["y_true"].device)]}
    res = pm.test_epoch_end([sub], quiet=True)
    n = int(ok.sum())
    acc, ndcg = mo.get_acc(y[ok], s64[ok])
    assert res["n"] == n
    for a, slot in (("acc1", 2), ("acc5", 1), ("acc10", 0), ("acc20", 3)):
        assert abs(res[a] - acc[slot, 0] / n) < 1e-12, a
        assert abs(res["ndcg" + a[3:]] - ndcg[slot, 0] / n) < 1e-9, a
    assert abs(res["mrr"] - mo.mrr_metric(y[ok], s64[ok]) / n) < 1e-9


class _Calls:
    """Records the libmobgt entry points ops calls (the dispatch check)."""

    def __init__(self, monkeypatch):
        from mobgt_b200 import _C
        self.names, real = [], _C.call

        def call(name, *a):
            self.names.append(name)
            return real(name, *a)
        monkeypatch.setattr(_C, "call", call)


@pytest.mark.gpu
@pytest.mark.parametrize("dataset_name", ["toyotagraph", "gowalla_nevda", "foursquaregraph"])
def test_precision32_eval_ranks_like_float64_oracle(lib_built, dataset_name, monkeypatch):
    from mobgt_b200 import model
    from test_round2_gpu import _pair
    w, items, om, pm, ob, pb = _pair(dataset_name, "c1", [(None, 24, 30, 9)], precision=32)
    calls = _Calls(monkeypatch)
    y_true = pb.y if dataset_name == "toyotagraph" else pb.y - 1
    _check_model_eval_vs_float64(pm, om, pb, ob, y_true)
    assert "mobgt_head_topk_f32" in calls.names and "mobgt_head_topk" not in calls.names
    model.ops.enable_tf32(True)


@pytest.mark.gpu
def test_precision32_eval_on_the_real_gowalla_batch(lib_built):
    from mobgt_b200 import collator, model, owndata
    world, splits = owndata.unpack_dataset(np.load(NPZ))
    items = [it for it in splits["train"][:80] if len(it.x) <= 96][:32]
    hp = dict(n_layers=6, num_heads=8, hidden_dim=128, dropout_rate=0.0, intput_dropout_rate=0.0, weight_decay=0.01, ffn_dim=1024,
              warmup_updates=10, tot_updates=100, peak_lr=2e-4, end_lr=1e-9, edge_type="multi_hop", multi_hop_max_dist=20,
              attention_dropout_rate=0.0)
    torch.manual_seed(5)
    om = mo.Graphormer(world, n_layers=6, ffn_dim=1024, dataset_name="gowalla_nevda", multi_hop_max_dist=20).eval()
    with torch.no_grad():
        for emb in (om.edge_encoder, om.rel_pos_encoder, om.poi_pos_encoder):
            emb.weight.mul_(0.3)
            emb.weight[0].zero_()
        om.edge_dis_encoder.weight.mul_(0.3)
    pm = model.Graphormer(dataset_name="gowalla_nevda", world=world, precision=32, **hp).cuda().eval()
    missing, _ = pm.load_state_dict(om.state_dict(), strict=False)
    assert not missing, missing
    ob = mo.collate([mo.preprocess_item(it, hop_cap=20) for it in items], world, multi_hop_max_dist=20, rel_pos_max=1024)
    pb = collator.collator_gowalla(items, max_node=512, multi_hop_max_dist=20, rel_pos_max=1024, world=world)
    _check_model_eval_vs_float64(pm, om, pb, ob, pb.y - 1)
    model.ops.enable_tf32(True)


@pytest.mark.gpu
def test_precision16_eval_keeps_the_bf16_head(lib_built, monkeypatch):
    from test_round2_gpu import _pair
    w, items, om, pm, ob, pb = _pair("gowalla_nevda", "tiny", [(None, 6, 12, 4)])
    assert pm.precision == 16
    calls = _Calls(monkeypatch)
    with torch.no_grad():
        out = pm.test_step(pb)
    assert out["rank"].dtype == torch.int32
    assert "mobgt_head_topk" in calls.names and "mobgt_head_topk_f32" not in calls.names


@pytest.mark.gpu
def test_entry_precision32_test_prints_the_oracle_metrics(lib_built, tmp_path, capsys):
    """`entry --precision 32 --test` from a checkpoint of oracle weights: the printed metric lines are those get_acc /
    MRR_metric give on the oracle's float64 logits of the same test items, batch by batch."""
    from mobgt_b200 import entry, model, synth
    seed, n_test, bs = 1, 24, 16
    w = synth.make_world("tiny", seed=seed, dataset_name="toyotagraph")
    test = synth.make_items(w, n_test, synth.CONFIGS["tiny"]["cap"], seed=seed, cfg_id=12, n_fixed=9)
    torch.manual_seed(7)
    om = mo.Graphormer(w, n_layers=2, ffn_dim=256, dataset_name="toyotagraph", multi_hop_max_dist=20).eval()
    with torch.no_grad():
        for emb in (om.edge_encoder, om.rel_pos_encoder, om.poi_pos_encoder):
            emb.weight.mul_(0.3)
            emb.weight[0].zero_()
        om.edge_dis_encoder.weight.mul_(0.3)
    ck = str(tmp_path / "oracle.ckpt")
    torch.save({"state_dict": om.state_dict()}, ck)
    args = ["--dataset_name", "toyotagraph", "--gpus", "1", "--precision", "32", "--batch_size", str(bs), "--hidden_dim", "128",
            "--num_heads", "8", "--n_layers", "2", "--ffn_dim", "256", "--edge_type", "multi_hop", "--seed", str(seed),
            "--synthetic", "tiny", "--train_graphs", "16", "--test_graphs", str(n_test), "--n_fixed", "9",
            "--multi_hop_max_dist", "20", "--test", "--checkpoint_path", ck, "--default_root_dir", str(tmp_path)]
    r = entry.cli_main(args)
    printed = [l for l in capsys.readouterr().out.splitlines() if l.startswith(("ACC", "NDCG", "MRR"))]
    tot = {k_: 0.0 for k_ in ("acc1", "acc5", "acc10", "ndcg1", "ndcg5", "ndcg10", "mrr")}
    for i in range(0, n_test, bs):
        ob = mo.collate([mo.preprocess_item(it, hop_cap=20) for it in test[i:i + bs]], w, multi_hop_max_dist=20, rel_pos_max=1024)
        z64, W64, b64 = _oracle64_z(om, ob)
        s64 = z64 @ W64.t() + b64
        y = ob.y.long().view(-1)
        s_t = s64.gather(1, y.view(-1, 1))
        gap = (s64 - s_t).abs()
        gap.scatter_(1, y.view(-1, 1), float("inf"))
        # fp32 mode is within 1e-5 x max |logit| of the oracle: no other logit within twice that of a target's, so no rank
        # can move and the 4-digit lines must be exact
        assert (gap.min(1).values > 2e-5 * s64.abs().max()).all()
        acc, ndcg = mo.get_acc(y, s64)
        for a, slot in (("1", 2), ("5", 1), ("10", 0)):
            tot["acc" + a] += acc[slot, 0]
            tot["ndcg" + a] += ndcg[slot, 0]
        tot["mrr"] += mo.mrr_metric(y, s64)
    avg = {k_: v / n_test for k_, v in tot.items()}
    assert r["metrics"]["n"] == n_test
    for k_ in avg:
        assert abs(r["metrics"][k_] - avg[k_]) < 1e-9, (k_, r["metrics"][k_], avg[k_])
    assert printed == [f"ACC @1: {round(avg['acc1'], 4)}, @5: {round(avg['acc5'], 4)}, @10: {round(avg['acc10'], 4)}",
                       f"NDCG @1: {round(avg['ndcg1'], 4)}, @5: {round(avg['ndcg5'], 4)}, @10: {round(avg['ndcg10'], 4)}",
                       f"MRR: {round(avg['mrr'], 4)}"]
    model.ops.enable_tf32(True)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_entry_precision32_eval_vocab_parallel_matches_one_rank(lib_built, tmp_path):
    """`entry --precision 32 --test --eval_vocab_parallel` on 2 ranks (out_proj sharded by vocabulary rows, fp32 head on each
    shard) prints the metrics of the 1-rank run of the same checkpoint."""
    import re
    import subprocess
    common = ["--dataset_name", "toyotagraph", "--accelerator", "ddp", "--precision", "32", "--batch_size", "16", "--hidden_dim",
              "128", "--num_heads", "8", "--n_layers", "2", "--ffn_dim", "256", "--edge_type", "multi_hop", "--multi_hop_max_dist",
              "20", "--seed", "1", "--max_epochs", "1", "--synthetic", "tiny", "--train_graphs", "32", "--test_graphs", "41",
              "--default_root_dir", str(tmp_path)]
    env = dict(os.environ, PYTHONPATH=ROOT)
    run1 = lambda extra: subprocess.run([sys.executable, "-m", "mobgt_b200.entry"] + common + extra, capture_output=True, text=True,
                                        env=env, cwd=ROOT, timeout=600)
    run2 = lambda extra: subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                                         "--master-addr", "127.0.0.1", "--master-port", "29579", "-m", "mobgt_b200.entry"] + common
                                        + extra, capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    tr = run1(["--limit_train_steps", "2"])
    assert tr.returncode == 0, tr.stderr[-2000:]
    ck = os.path.join(str(tmp_path), "lightning_logs", "checkpoints", "last.ckpt")
    a = run1(["--test", "--checkpoint_path", ck])
    b = run2(["--test", "--eval_vocab_parallel", "--checkpoint_path", ck])
    assert a.returncode == 0 and b.returncode == 0, (a.stderr[-1500:], b.stderr[-1500:])
    nums = lambda out: [float(x) for line in out.splitlines() if line.startswith(("ACC", "NDCG", "MRR")) for x in re.findall(r"[-+]?\d*\.\d+", line)]
    na, nb = nums(a.stdout), nums(b.stdout)
    assert len(na) == 7 and len(nb) == 7, (a.stdout, b.stdout)
    # each rank encodes its own graphs (other GEMM shapes: last-bit differences may flip a near tie), as the bf16 2-rank test
    assert all(abs(x - y) <= 2e-3 for x, y in zip(na, nb)), (na, nb)
